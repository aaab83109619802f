// TEST INFRASTRUCTURE ONLY -- the conjunction screening sources (conjunction_kernel.cuh: the per-interval functions and
// the pre-pass kernel) of the host build, on top of the wrappers of hostk_main.cpp.  Built by
// tests/test_conjunctions_host.py next to libmpc_hostk.so; the threads of a launch run one after the other.  The pair
// kernel (warp collectives, a CTA barrier) is device-only: hostk_conj_screen runs its per-pair work, the sphere filter and
// conj_interval, over every pair i < j and interval in a plain loop.
#include "hostk_main.cpp"
#include "conjunction_kernel.cuh"

// the pre-pass: y [n][7][T], scale [n][2] -> X [T][6][n], S [T-1][4][n], skipped [n] (zeroed here)
extern "C" void hostk_conj_prepass(const double *y, const double *scale, int n, int T, double h, double *X, double *S,
                                   int32_t *skipped)
{
    for (int s = 0; s < n; ++s) skipped[s] = 0;
    run_grid((long long)n * T, [&] { mpc::conj_prepass_kernel<kBlock>(y, scale, n, T, h, X, S, skipped); });
}

// conj_sphere of m segments: q0, q1 [m][6] -> out [m][4]
extern "C" void hostk_conj_sphere(const double *q0, const double *q1, int m, double h, double *out)
{
    for (int e = 0; e < m; ++e) mpc::conj_sphere(q0 + 6 * e, q1 + 6 * e, h, out + 4 * e);
}

// conj_interval of m pair-intervals: q [m][4][6] (qi0, qi1, qj0, qj1), fl [m] (bit 0: first, bit 1: last) ->
// ev [m][kConjMaxEv][4] (s, d, v, flags), n [m]
extern "C" int hostk_conj_interval(const double *q, const int32_t *fl, int m, double h, double thr, double *ev, int32_t *n)
{
    for (int e = 0; e < m; ++e) {
        mpc::ConjEvent buf[mpc::kConjMaxEv];
        const double *p = q + 24 * e;
        n[e] = mpc::conj_interval(p, p + 6, p + 12, p + 18, h, thr, fl[e] & 1, (fl[e] >> 1) & 1, buf);
        for (int k = 0; k < n[e]; ++k) {
            double *o = ev + ((size_t)e * mpc::kConjMaxEv + k) * 4;
            o[0] = buf[k].s;
            o[1] = buf[k].d;
            o[2] = buf[k].v;
            o[3] = buf[k].flags;
        }
    }
    return mpc::kConjMaxEv;
}

// the whole screen: pre-pass, then every pair i < j and interval through the sphere filter and conj_interval, the
// events as the pair kernel records them.  counters [3]: events found, events flagged, pair-intervals past the filter.
extern "C" void hostk_conj_screen(const double *y, const double *scale, int n, int T, double h, double thr, double *X,
                                  double *S, int32_t *skipped, mpc::ConjRecord *out, long long capacity,
                                  long long *counters)
{
    hostk_conj_prepass(y, scale, n, T, h, X, S, skipped);
    counters[0] = counters[1] = counters[2] = 0;
    for (int i = 0; i < n; ++i)
        for (int j = i + 1; j < n; ++j)
            for (int k = 0; k < T - 1; ++k) {
                const double *si = S + (size_t)k * 4 * n, *sj = si;
                const double dx = si[i] - sj[j], dy = si[n + i] - sj[n + j], dz = si[2 * n + i] - sj[2 * n + j];
                const double R = si[3 * n + i] + sj[3 * n + j] + thr;
                if (!(dx * dx + dy * dy + dz * dz <= R * R)) continue;
                ++counters[2];
                double q[4][6];
                for (int c = 0; c < 6; ++c) {
                    q[0][c] = X[((size_t)k * 6 + c) * n + i];
                    q[1][c] = X[((size_t)(k + 1) * 6 + c) * n + i];
                    q[2][c] = X[((size_t)k * 6 + c) * n + j];
                    q[3][c] = X[((size_t)(k + 1) * 6 + c) * n + j];
                }
                mpc::ConjEvent ev[mpc::kConjMaxEv];
                const int m = mpc::conj_interval(q[0], q[1], q[2], q[3], h, thr, k == 0, k == T - 2, ev);
                for (int e = 0; e < m; ++e) {
                    if (ev[e].flags) ++counters[1];
                    if (counters[0] < capacity)
                        out[counters[0]] = mpc::ConjRecord{i, j, k, ev[e].flags, fma((double)k, h, ev[e].s * h), ev[e].d, ev[e].v};
                    ++counters[0];
                }
            }
}
