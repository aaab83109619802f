/*
 * TEST INFRASTRUCTURE ONLY -- the plain-C oracle's RK45 propagation (oracle/mpc_oracle.c, included here unchanged for its
 * controller laws, tableau and helpers) with the drag under an altitude-dependent density: the Chebyshev series of
 * log rho in log h of mpc_atmosphere (include/mpc_b200.h), evaluated at h = |r| R0 - r_earth.  Built and bound by
 * tests/atmo_oracle.py; never linked by the product library.
 */
#include "../oracle/mpc_oracle.c"

/* An altitude-dependent density of the propagator's drag (the layout of mpc_atmosphere, include/mpc_b200.h): log rho as
 * sum_k coef[k] T_k(t), t = (log h - (log h_min + log h_max) / 2) / ((log h_max - log h_min) / 2), h = |r| R0 - r_earth. */
typedef struct {
    double h_min, h_max, r_earth;
    int n, reserved;
    double coef[32];
} orc_atmo;

/* rho(h) of the series; *out = 1 when h is outside [h_min, h_max] */
static double atmo_rho(const orc_atmo *a, double h, int *out)
{
    const double lo = log(a->h_min), hi = log(a->h_max);
    const double t = (log(h) - 0.5 * (lo + hi)) / (0.5 * (hi - lo));
    double b1 = 0.0, b2 = 0.0;
    for (int k = a->n - 1; k >= 1; --k) {
        const double b = 2.0 * t * b1 - b2 + a->coef[k];
        b2 = b1;
        b1 = b;
    }
    *out = (h < a->h_min || h > a->h_max);
    return exp(t * b1 - b2 + a->coef[0]);
}

/* f / tf : simulator.py:130-160; atmo != NULL: the drag's density rho(h) instead of RHO_ATM (returns 2 outside its range) */
static int dyn_atmo(const double *y, const double *u, const orc_params *p, int drag, int j2, const orc_atmo *atmo, double *dy)
{
    int out = 0;
    const double *r = y, *v = y + 3;
    double m = y[6];
    if (!(m > 0.0)) return 1;
    double rn = norm3(r);
    double g = -p->MU / (rn * rn * rn);
    for (int i = 0; i < 3; ++i) {
        dy[i] = v[i];
        dy[3 + i] = g * r[i] + u[i] / m;
    }
    if (drag) {
        double vn = norm3(v);
        double rho = atmo ? atmo_rho(atmo, rn * p->R0 - atmo->r_earth, &out) : p->RHO_ATM;
        double c = -0.5 * p->C_D * p->S * (1.0 / m) * (rho / p->RHO) * vn;
        for (int i = 0; i < 3; ++i) dy[3 + i] += c * v[i];
    }
    if (j2) {
        double q = 5.0 * (r[2] / rn) * (r[2] / rn);
        double k = 1.5 * p->J2 * p->MU * p->R_E * p->R_E / pow(rn, 5);
        dy[3] += k * (q - 1.0) * r[0];
        dy[4] += k * (q - 1.0) * r[1];
        dy[5] += k * (q - 3.0) * r[2];
    }
    dy[6] = -norm3(u) / (p->G0 * p->ISP);
    return out ? 2 : 0;
}

static int prop_rhs_atmo(const double *y, double tau, double tf, const orc_params *p, int kind, const double *cp,
                         const double *tab, int Ku, double end_tau, const orc_atmo *atmo, double *dy)
{
    double u[3];
    ctrl_eval(kind, cp, tab, Ku, end_tau, y, tau, u);
    int st = dyn_atmo(y, u, p, p->include_drag, p->include_J2, atmo, dy);
    if (st) return st;
    for (int i = 0; i < 7; ++i) dy[i] *= tf;
    return 0;
}

/* orc_propagate_rk45 (the C restatement of the reference's solve_ivp call, statement for statement) with the drag
 * under *atmo; status 2: an altitude outside its range (the run ends there, as at a non-positive mass, status 1) */
int orc_propagate_rk45_atmo(const double *y0, const double *tf, const orc_params *p, int kind, const double *cp,
                          const double *ctrl_tab, int Ku, int tab_per_sat, double end_tau, const double *end_tau_arr, int N,
                          int T, double rtol, double atol, double max_step, double *y_out, double *u_out, int *status,
                          int *n_steps, int *n_rej, int nthreads, const orc_atmo *atmo)
{
    int bad = 0;
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel for schedule(static) reduction(+ : bad)
    for (int s = 0; s < N; ++s) {
        const double *tab = ctrl_tab ? ctrl_tab + (tab_per_sat ? (long)s * 3 * Ku : 0) : 0;
        const double et = end_tau_arr ? end_tau_arr[s] : end_tau;
        const double tfs = tf[s], t_bound = 1.0;
        double y[7], f[7], K[7][7], ynew[7], fnew[7], tmp[7], sc[7], us[3];
        int st = 0, steps = 0, rej = 0;
        for (int c = 0; c < 7; ++c) y[c] = y0[s * 7 + c];
        double t = 0.0;
        /* np.linspace(0, 1, T): arange(T) * step, last point exactly 1 */
        const double lstep = (T > 1) ? 1.0 / (double)(T - 1) : 0.0;
#define TEVAL(j) (((j) == T - 1 && T > 1) ? 1.0 : (double)(j) * lstep)
        int ti = 0;
        st |= prop_rhs_atmo(y, t, tfs, p, kind, cp, tab, Ku, et, atmo, f);
        double h_abs = 0.0;
        if (!st) { /* select_initial_step */
            double interval_length = fabs(t_bound - t);
            for (int i = 0; i < 7; ++i) sc[i] = atol + fabs(y[i]) * rtol;
            for (int i = 0; i < 7; ++i) tmp[i] = y[i] / sc[i];
            double d0 = rms7(tmp);
            for (int i = 0; i < 7; ++i) tmp[i] = f[i] / sc[i];
            double d1 = rms7(tmp);
            double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
            if (h0 > interval_length) h0 = interval_length;
            for (int i = 0; i < 7; ++i) ynew[i] = y[i] + h0 * f[i];
            st |= prop_rhs_atmo(ynew, t + h0, tfs, p, kind, cp, tab, Ku, et, atmo, fnew);
            for (int i = 0; i < 7; ++i) tmp[i] = (fnew[i] - f[i]) / sc[i];
            double d2 = rms7(tmp) / h0;
            double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : pow(0.01 / fmax(d1, d2), 1.0 / 5.0);
            h_abs = fmin(fmin(100 * h0, h1), fmin(interval_length, max_step));
        }
        while (!st && t < t_bound) {
            double min_step = 10 * fabs(nextafter(t, INFINITY) - t);
            if (h_abs > max_step) h_abs = max_step;
            else if (h_abs < min_step) h_abs = min_step;
            int accepted = 0, rejected = 0;
            double t_new = t, h = 0.0;
            while (!accepted && !st) {
                if (h_abs < min_step) {
                    st = 4;
                    break;
                }
                h = h_abs;
                t_new = t + h;
                if (t_new - t_bound > 0) t_new = t_bound;
                h = t_new - t;
                h_abs = fabs(h);
                memcpy(K[0], f, sizeof f);
                for (int q = 1; q < 6 && !st; ++q) {
                    for (int i = 0; i < 7; ++i) {
                        double dy = 0.0;
                        for (int l = 0; l < q; ++l) dy += K[l][i] * DP_A[q][l];
                        tmp[i] = y[i] + dy * h;
                    }
                    st |= prop_rhs_atmo(tmp, t + DP_C[q] * h, tfs, p, kind, cp, tab, Ku, et, atmo, K[q]);
                }
                if (st) break;
                for (int i = 0; i < 7; ++i) {
                    double d = 0.0;
                    for (int l = 0; l < 6; ++l) d += K[l][i] * DP_B[l];
                    ynew[i] = y[i] + h * d;
                }
                st |= prop_rhs_atmo(ynew, t + h, tfs, p, kind, cp, tab, Ku, et, atmo, fnew);
                if (st) break;
                memcpy(K[6], fnew, sizeof fnew);
                for (int i = 0; i < 7; ++i) {
                    double e = 0.0;
                    for (int l = 0; l < 7; ++l) e += K[l][i] * DP_E[l];
                    tmp[i] = e * h / (atol + fmax(fabs(y[i]), fabs(ynew[i])) * rtol);
                }
                double err = rms7(tmp);
                if (err < 1.0) {
                    double factor = (err == 0.0) ? 10.0 : fmin(10.0, 0.9 * pow(err, -0.2));
                    if (rejected && factor > 1.0) factor = 1.0;
                    h_abs *= factor;
                    accepted = 1;
                } else {
                    h_abs *= fmax(0.2, 0.9 * pow(err, -0.2));
                    rejected = 1;
                    ++rej;
                }
            }
            if (st) break;
            ++steps;
            /* samples with t_eval <= t_new, off the dense output of this step */
            if (ti < T && TEVAL(ti) <= t_new) {
                double Q[7][4];
                for (int i = 0; i < 7; ++i)
                    for (int m = 0; m < 4; ++m) {
                        double q = 0.0;
                        for (int l = 0; l < 7; ++l) q += K[l][i] * DP_P[l][m];
                        Q[i][m] = q;
                    }
                while (ti < T && TEVAL(ti) <= t_new) {
                    double te = TEVAL(ti), xx = (te - t) / h, pw[4], ys[7];
                    pw[0] = xx;
                    for (int m = 1; m < 4; ++m) pw[m] = pw[m - 1] * xx;
                    for (int i = 0; i < 7; ++i) {
                        double q = 0.0;
                        for (int m = 0; m < 4; ++m) q += Q[i][m] * pw[m];
                        ys[i] = h * q + y[i];
                        y_out[((long)s * 7 + i) * T + ti] = ys[i];
                    }
                    if (u_out) { /* extract_uk, linearize_discretize.py:393-411 */
                        ctrl_eval(kind, cp, tab, Ku, et, ys, te, us);
                        for (int c = 0; c < 3; ++c) u_out[((long)s * 3 + c) * T + ti] = us[c];
                    }
                    ++ti;
                }
            }
            memcpy(y, ynew, sizeof y);
            memcpy(f, fnew, sizeof f);
            t = t_new;
            if (steps > 50000000) st = 4;
        }
#undef TEVAL
        if (st) { /* the reference raises: nothing is returned for this satellite */
            for (int j = ti; j < T; ++j) {
                for (int i = 0; i < 7; ++i) y_out[((long)s * 7 + i) * T + j] = NAN;
                if (u_out)
                    for (int c = 0; c < 3; ++c) u_out[((long)s * 3 + c) * T + j] = NAN;
            }
        }
        if (status) status[s] = st;
        if (n_steps) n_steps[s] = steps;
        if (n_rej) n_rej[s] = rej;
        bad += (st != 0);
    }
    return bad;
}

