// mpc_b200.cu -- C-ABI (include/mpc_b200.h) over the sm_100a kernels.  No CPU fallback: every entry
// point either launches CUDA work or returns an error.
#include "../../include/mpc_b200.h"

#include <cuda.h>   // types of the stream memory operations only; the entry point is fetched at run time
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <limits>
#include <vector>

#include <math_constants.h>

#include "discretize_kernel.cuh"
#include "discretize_adaptive_kernel.cuh"
#include "discretize_default_kernel.cuh"
#include "propagate_kernel.cuh"
#include "propagate_rk45_kernel.cuh"
#include "mpc_b200_drag.h"
#include "mpc_b200_units.h"
#include "mpc_b200_shard.h"
#include "mpc_b200_atmo.h"
#include "mpc_b200_rk23.h"
#include "mpc_b200_conj.h"
#include "constraint_terms_kernel.cuh"
#include "discretize_drag_kernel.cuh"
#include "discretize_pair_kernel.cuh"
#include "discretize_group_kernel.cuh"

namespace {

thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                                       \
    do {                                                                                                     \
        cudaError_t e_ = (expr);                                                                             \
        if (e_ != cudaSuccess) return fail(MPC_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                                           __FILE__, __LINE__);                                              \
    } while (0)

constexpr int kDiscBlock = 128;
constexpr int kPropBlock = 32;
constexpr int kPropBlockOverlap = 128;

mpc::DiscParams disc_params(const mpc_params *p)
{
    mpc::DiscParams d;
    d.mu = p->mu;
    d.kj2 = 1.5 * p->j2 * p->mu * p->r_e * p->r_e;
    d.inv_ve = 1.0 / (p->g0 * p->isp);
    return d;
}

mpc::PropParams prop_params(const mpc_params *p)
{
    mpc::PropParams d;
    d.mu = p->mu;
    d.kj2 = 1.5 * p->j2 * p->mu * p->r_e * p->r_e;
    d.inv_ve = 1.0 / (p->g0 * p->isp);
    d.drag_k = p->include_drag ? 0.5 * p->c_d * p->s_area * (p->rho_atm / p->rho) : 0.0;
    d.include_j2 = p->include_j2;
    d.include_drag = p->include_drag;
    return d;
}

// ---- altitude-dependent atmosphere (mpc_propagate_batch_rk45_atmo) ----------------------------------------------------
// The kernel constants of a satellite under the atmosphere: drag_k without the density (rho(h) multiplies it in the
// kernel) and the metres per unit length of its constants, r_earth / r_e
mpc::PropParams atmo_prop_params(const mpc_params *p)
{
    mpc::PropParams d = prop_params(p);
    d.drag_k = 0.5 * p->c_d * p->s_area / p->rho;
    return d;
}

mpc::AtmoSat atmo_sat(const mpc_params *q, double r_earth)
{
    mpc::AtmoSat a;
    a.P = atmo_prop_params(q);
    a.len = r_earth / q->r_e;
    return a;
}

mpc::AtmoParams atmo_params(const mpc_atmosphere *a, double len)
{
    mpc::AtmoParams A{};
    for (int k = 0; k < a->n; ++k) A.coef[k] = a->coef[k];
    A.n = a->n;
    const double lo = std::log(a->h_min), hi = std::log(a->h_max);
    A.s_mid = 0.5 * (lo + hi);
    A.s_ihalf = 2.0 / (hi - lo);
    A.h_min = a->h_min;
    A.h_max = a->h_max;
    A.r_earth = a->r_earth;
    A.len = len;
    return A;
}

bool positive(double x) { return std::isfinite(x) && x > 0.0; }

// the model, and what the drag under it divides by (r_e for the length unit, rho), of p or of every consts[s]
int check_atmo(const mpc_atmosphere *a, const mpc_params *p, const mpc_sat_consts *c, int n)
{
    if (!a || !p) return fail(MPC_E_INVALID, "null atmosphere / params");
    if (!p->include_drag) return fail(MPC_E_INVALID, "an atmosphere is the density of the drag: it needs include_drag");
    if (a->n < 1 || a->n > MPC_RHO_CHEB) return fail(MPC_E_INVALID, "atmosphere: need 1 <= n <= %d (got %d)", MPC_RHO_CHEB, a->n);
    if (!positive(a->h_min) || !(std::isfinite(a->h_max) && a->h_max > a->h_min))
        return fail(MPC_E_INVALID, "atmosphere: need 0 < h_min < h_max (got %g, %g)", a->h_min, a->h_max);
    if (!positive(a->r_earth)) return fail(MPC_E_INVALID, "atmosphere: need r_earth > 0 (got %g)", a->r_earth);
    for (int k = 0; k < a->n; ++k)
        if (!std::isfinite(a->coef[k])) return fail(MPC_E_INVALID, "atmosphere: coef[%d] is not finite", k);
    if (!std::isfinite(p->c_d) || !std::isfinite(p->s_area)) return fail(MPC_E_INVALID, "need finite c_d and s_area");
    if (!c) {
        if (!positive(p->r_e) || !positive(p->rho))
            return fail(MPC_E_INVALID, "an atmosphere needs r_e > 0 and rho > 0 (got %g, %g)", p->r_e, p->rho);
        return MPC_SUCCESS;
    }
    for (int s = 0; s < n; ++s)
        if (!positive(c[s].r_e) || !positive(c[s].rho))
            return fail(MPC_E_INVALID, "consts[%d]: an atmosphere needs r_e > 0 and rho > 0 (got %g, %g)", s, c[s].r_e, c[s].rho);
    return MPC_SUCCESS;
}

// ---- per-satellite designer units (the *_units entry points) ---------------------------------------------------------
static_assert(sizeof(mpc::AtmoSat) <= MPC_SAT_SCRATCH_DOUBLES * sizeof(double), "per-satellite scratch too small");
static_assert(sizeof(mpc::PropParams) <= MPC_SAT_SCRATCH_DOUBLES * sizeof(double) &&
              sizeof(mpc::DiscParams) <= MPC_SAT_SCRATCH_DOUBLES * sizeof(double), "per-satellite scratch too small");

int check_sat_consts(const mpc_sat_consts *c, int n)
{
    if (!c) return fail(MPC_E_INVALID, "null consts");
    for (int s = 0; s < n; ++s) {
        const double v[7] = {c[s].mu, c[s].r_e, c[s].j2, c[s].g0, c[s].isp, c[s].s_area, c[s].rho};
        for (double x : v)
            if (!std::isfinite(x)) return fail(MPC_E_INVALID, "consts[%d]: every value must be finite", s);
        if (!(c[s].mu > 0.0) || !(c[s].g0 * c[s].isp > 0.0))
            return fail(MPC_E_INVALID, "consts[%d]: need mu > 0 and g0 * isp > 0 (got %g, %g)", s, c[s].mu, c[s].g0 * c[s].isp);
    }
    return MPC_SUCCESS;
}

// q (a copy of the launch's mpc_params) with satellite s's per-scale fields: its kernel constants come out of
// disc_params / prop_params themselves, the expressions (and so the bits) of a single-constant launch under consts[s]
void with_consts(mpc_params &q, const mpc_sat_consts &c)
{
    q.mu = c.mu;
    q.r_e = c.r_e;
    q.j2 = c.j2;
    q.g0 = c.g0;
    q.isp = c.isp;
    q.s_area = c.s_area;
    q.rho = c.rho;
}

// derive the kernel constants of every satellite and copy them into the device scratch (the vector is pageable:
// cudaMemcpyAsync has staged it when it returns)
template <typename T, typename F>
int upload_sat_table(const mpc_params *p, const mpc_sat_consts *c, int n, void *scratch, cudaStream_t st, F derive)
{
    if (!scratch) return fail(MPC_E_INVALID, "null consts_scratch");
    if (mpc_units_sizeof(0) != sizeof(mpc::DiscParams) || mpc_units_sizeof(1) != sizeof(mpc::DstTab) ||
        mpc_units_sizeof(2) != sizeof(mpc::PropParams) || mpc_units_sizeof(3) != sizeof(mpc::CtrlParams) ||
        mpc_units_sizeof(4) != sizeof(mpc::Rk45Opts))
        return fail(MPC_E_CUDA, "mpc_b200_units.cu was built against different parameter structs");
    if (mpc_atmo_sizeof(0) != sizeof(mpc::PropParams) || mpc_atmo_sizeof(1) != sizeof(mpc::CtrlParams) ||
        mpc_atmo_sizeof(2) != sizeof(mpc::Rk45Opts) || mpc_atmo_sizeof(3) != sizeof(mpc::AtmoParams) ||
        mpc_atmo_sizeof(4) != sizeof(mpc::AtmoSat))
        return fail(MPC_E_CUDA, "mpc_b200_atmo.cu was built against different parameter structs");
    std::vector<T> v((size_t)n);
    mpc_params q = *p;
    for (int s = 0; s < n; ++s) {
        with_consts(q, c[s]);
        v[s] = derive(&q);
    }
    CUDA_TRY(cudaMemcpyAsync(scratch, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
    return MPC_SUCCESS;
}

std::atomic<int> g_tuning{0};
std::atomic<int> g_gather_skip_const{0}, g_gather_stagger{0};   // mpc_set_gather_tuning
// Options of one mpc_*_gather call (layout, what to send, how to start), visible to the launchers for its duration --
// per call and per thread, unlike the process-wide knobs of mpc_set_gather_tuning (kept for the older entry points).
struct GatherCall {
    bool active = false;
    int skip_const = 0, stagger = 0;
    long long km_ntot = 0, km_soff = 0;
};
thread_local GatherCall g_gather;
struct GatherScope {
    explicit GatherScope(const GatherCall &g) { g_gather = g; }
    ~GatherScope() { g_gather = GatherCall(); }
};
thread_local int g_ucols = 0;  // columns of u when it lives on its own grid (set by the *_ugrid entry points)
struct UcolsScope {            // routes the launchers to the general-grid input hold for the duration of one call
    explicit UcolsScope(int n) { g_ucols = n; }
    ~UcolsScope() { g_ucols = 0; }
};

template <bool J2, int BLOCK, int MAXREG, int NDST, bool GENU = false>
int launch_disc_cfg(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                    int n_sub, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status,
                    cudaStream_t st)
{
    auto kern = mpc::discretize_kernel<J2, BLOCK, MAXREG, NDST, GENU>;
    const size_t smem = (size_t)mpc::kDiscSlots * BLOCK * sizeof(double);
    static thread_local int configured_dev = -1;
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (configured_dev != dev) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        configured_dev = dev;
    }
    const long long n_int = (long long)n_sats * (K - 1);
    const unsigned grid = (unsigned)((n_int + BLOCK - 1) / BLOCK);
    kern<<<grid, BLOCK, smem, st>>>(x, u, tf, P, n_sats, K, g_ucols, n_sub, dst, pitch, offset, status);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

// discretize_pair_kernel: integrator steps spanning two quadrature nodes (needs an even number of panels)
// mpc_set_tuning(37 / 38): the 21-node Euler-Maclaurin form of the 101-node trapezoid sums off / on (kEmW)
std::atomic<int> g_em{1};
// mpc_set_tuning(39 / 40): the 11-node form on fifth-order steps (kEmW3) off / on, for the intervals of the 21-node form
std::atomic<int> g_em3{1};
int em_level() { return g_em.load(std::memory_order_relaxed) ? 1 + g_em3.load(std::memory_order_relaxed) : 0; }

template <bool J2, int BLOCK, int MAXREG, int NDST>
int launch_pair_cfg(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                    int n_sub, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status,
                    cudaStream_t st, int k0 = 0, int kc = -1)
{
    if (kc < 0) kc = K - 1;   // the whole batch
    auto kern = mpc::discretize_pair_kernel<J2, BLOCK, MAXREG, NDST>;
    const size_t smem = (size_t)mpc::kDiscSlots * BLOCK * sizeof(double);
    static thread_local int configured_dev = -1;
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (configured_dev != dev) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        configured_dev = dev;
    }
    const long long n_int = (long long)n_sats * kc;
    const unsigned grid = (unsigned)((n_int + BLOCK - 1) / BLOCK);
    mpc::DstTab tab = dst;
    tab.em = em_level();
    kern<<<grid, BLOCK, smem, st>>>(x, u, tf, P, n_sats, K, n_sub, tab, pitch, offset, status, k0, kc, nullptr, nullptr);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

std::atomic<int> g_pair{1};   // mpc_set_tuning(7) switches the two-node steps off (one step per node everywhere)
std::atomic<int> g_host_windows{32};   // mpc_set_tuning(26..29): k-windows of the streamed host pass 16 / 32 / 48 / 64
std::atomic<int> g_group{1};  // mpc_set_tuning(23 / 24): the 8-lanes-per-interval kernel for small batches off / on
// Below this many intervals the thread-group mapping wins (measured on a B200, profiles/r02_x_small_batches.txt, both
// kernels with the 21-node form of the 101-node sums): the one-thread kernel needs 0.053 ms whatever the batch, the group
// kernel 0.044 ms up to ~1000 intervals, 0.049 ms at 2376 and 0.065 ms at 6336, where its 8x as many warps queue up on
// the schedulers.  (With all 101 nodes evaluated the numbers were 0.118 / 0.064 / 0.086 / 0.12 ms, r02_f_small_batches.)
constexpr long long kGroupMaxIntervals = 2560;

template <bool J2>
int launch_group(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                 int n_sub, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status, cudaStream_t st)
{
    constexpr int BLOCK = 32;                       // 4 intervals per CTA: spreads a small batch over every SM
    const long long n_int = (long long)n_sats * (K - 1);
    const unsigned grid = (unsigned)((n_int * 8 + BLOCK - 1) / BLOCK);
    mpc::DstTab tab = dst;
    tab.em = em_level();
    mpc::discretize_group_kernel<J2, BLOCK><<<grid, BLOCK, 0, st>>>(x, u, tf, P, n_sats, K, n_sub, tab, pitch, offset, status);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

// The production configuration plus the experimental ones mpc_set_tuning() selects (single destination,
// no J2 only: they exist to measure occupancy / register-cap trade-offs, see DESIGN.md).
template <bool J2, int NDST>
int launch_disc_n(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                  int n_sub, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status,
                  cudaStream_t st)
{
#define MPC_ARGS x, u, tf, P, n_sats, K, n_sub, dst, pitch, offset, status, st
    if (NDST == 1 && g_ucols > 0) return launch_disc_cfg<J2, kDiscBlock, 255, 1, true>(MPC_ARGS);
    if (!J2 && NDST == 1) {
        switch (g_tuning.load(std::memory_order_relaxed)) {
            case 1: return launch_disc_cfg<false, 32, 224, 1>(MPC_ARGS);   //  9 warps / SM
            case 2: return launch_disc_cfg<false, 64, 200, 1>(MPC_ARGS);   // 10 warps / SM
            case 3: return launch_disc_cfg<false, 32, 184, 1>(MPC_ARGS);   // 11 warps / SM
            case 4: return launch_disc_cfg<false, 64, 168, 1>(MPC_ARGS);   // 12 warps / SM
            case 5: return launch_disc_cfg<false, 64, 255, 1>(MPC_ARGS);   //  8 warps / SM, smaller CTAs
            case 6: return launch_disc_cfg<false, 256, 255, 1>(MPC_ARGS);  // one 8-warp CTA / SM
            default: break;
        }
    }
    // Small batches (BASELINE configs 1-2: 49 ... 6,336 intervals) cannot fill 148 SMs with 128-thread CTAs:
    // one-warp CTAs spread them over as many SMs as possible (same code, 224-register build, 9 CTAs/SM).
    // two quadrature nodes per integrator step where that is accurate (decided per thread inside the kernel)
    const bool pair = (g_ucols == 0) && g_pair.load(std::memory_order_relaxed);
    const long long n_int = (long long)n_sats * (K - 1);
    // north_star's "warp or thread-group per interval" for batches below one wave: 8 lanes per interval
    const int grp = g_group.load(std::memory_order_relaxed);   // 2: at any batch size (measurements)
    if (NDST == 1 && pair && dst.km_ntot == 0 && grp && (n_int <= kGroupMaxIntervals || grp == 2))
        return launch_group<J2>(MPC_ARGS);
    // more warps than SMs but at most one 4-warp CTA per SM: one warp per scheduler on every SM (one-warp CTAs of such a
    // batch land several to a scheduler: 0.27 instead of 0.115 ms on 15,104 intervals)
    if (NDST == 1 && pair && n_int > 148LL * 32 && n_int <= 148LL * 128)
        return launch_pair_cfg<J2, kDiscBlock, 255, 1>(MPC_ARGS);
    if (NDST == 1 && n_int < 148LL * 9 * 32 * 2)
        return pair ? launch_pair_cfg<J2, 32, 255, 1>(MPC_ARGS) : launch_disc_cfg<J2, 32, 224, 1>(MPC_ARGS);
    return pair ? launch_pair_cfg<J2, kDiscBlock, 255, NDST>(MPC_ARGS) : launch_disc_cfg<J2, kDiscBlock, 255, NDST>(MPC_ARGS);
#undef MPC_ARGS
}

template <bool J2>
int launch_disc(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                int n_sub, const mpc::DstTab &dst, int n_dst, long long pitch, long long offset, int32_t *status,
                cudaStream_t st)
{
    switch (n_dst) {
        case 1: return launch_disc_n<J2, 1>(x, u, tf, P, n_sats, K, n_sub, dst, pitch, offset, status, st);
        case 2: return launch_disc_n<J2, 2>(x, u, tf, P, n_sats, K, n_sub, dst, pitch, offset, status, st);
        case 4: return launch_disc_n<J2, 4>(x, u, tf, P, n_sats, K, n_sub, dst, pitch, offset, status, st);
        case 8: return launch_disc_n<J2, 8>(x, u, tf, P, n_sats, K, n_sub, dst, pitch, offset, status, st);
        default: return fail(MPC_E_INVALID, "n_dst must be 1, 2, 4 or 8 (got %d)", n_dst);
    }
}

struct AdaptiveOpts {   // scipy solve_ivp(RK45) controls of the reference's default quadrature mode
    double rtol, atol, max_step;
    int32_t *n_nodes;
    int drag = 0;           // drag branch of the linearisation (set from mpc_params by with_drag)
    double kf = 0.0;
    mpc::DragLin lin{};     // density model of the Jacobian's drag terms
    int rk23 = 0;           // scipy's RK23 in place of RK45 (mpc_discretize_batch_rk23[_host]; mpc_b200_rk23.cu)
};

template <bool J2, bool GENU>
int launch_adaptive_g(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                      const AdaptiveOpts &o, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status,
                      cudaStream_t st);

template <bool J2>
int launch_adaptive(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                    const AdaptiveOpts &o, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status,
                    cudaStream_t st)
{
    return g_ucols > 0 ? launch_adaptive_g<J2, true>(x, u, tf, P, n_sats, K, o, dst, pitch, offset, status, st)
                       : launch_adaptive_g<J2, false>(x, u, tf, P, n_sats, K, o, dst, pitch, offset, status, st);
}

std::atomic<int> g_default_v1{0};   // mpc_set_tuning(9): the round-1 build of the default-mode kernel (A/B measurements)

// The kernels of the drag branch live in mpc_b200_drag.cu (see there for why); this is the call across.
int launch_drag_unit(bool adaptive, int variant, int block, const double *x, const double *u, const double *tf,
                     const mpc::DiscParams &P, bool j2, double kf, const mpc::DragLin &L, int n_sats, int K, int n_sub,
                     double rtol, double atol, double max_step, const mpc::DstTab &dst, long long pitch, long long offset,
                     int32_t *status, int32_t *n_nodes, cudaStream_t st, bool drag = true, int ucols = 0)
{
    if (mpc_drag_sizeof(0) != sizeof(mpc::DiscParams) || mpc_drag_sizeof(1) != sizeof(mpc::DstTab) ||
        mpc_drag_sizeof(2) != sizeof(mpc::DragLin))
        return fail(MPC_E_CUDA, "mpc_b200_drag.cu was built against different parameter structs");
    MpcDragLaunch a{};
    a.x = x;
    a.u = u;
    a.tf = tf;
    a.disc_params = &P;
    a.dst_tab = &dst;
    a.drag_lin = &L;
    a.kf = kf;
    a.include_j2 = j2;
    a.n_sats = n_sats;
    a.K = K;
    a.n_sub = n_sub;
    a.variant = variant;
    a.block = block;
    a.drag = drag;
    a.ucols = ucols;
    a.rtol = rtol;
    a.atol = atol;
    a.max_step = max_step;
    a.pitch = pitch;
    a.offset = offset;
    a.status = status;
    a.n_nodes = n_nodes;
    a.stream = st;
    CUDA_TRY(adaptive ? mpc_drag_launch_adaptive(&a) : mpc_drag_launch_fixed(&a));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return MPC_SUCCESS;
}

template <typename Kern>
int configure_smem(Kern kern, size_t smem, int &configured_dev)
{
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (configured_dev != dev) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        configured_dev = dev;
    }
    return MPC_SUCCESS;
}

// round-1 build: Phi and its candidate in shared memory (52 KiB per warp), both ends of every panel evaluated
template <bool J2, bool GENU, bool DRAG>
int launch_adaptive_v1(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                       const AdaptiveOpts &o, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status,
                       cudaStream_t st)
{
    constexpr int BLOCK = 32;
    if (DRAG && (o.lin.n_rho > 1 || o.lin.n_drho > 0))
        return fail(MPC_E_UNSUPPORTED, "the round-1 default-mode kernel (mpc_set_tuning(9)) linearizes drag for a constant density only");
    // (kept for A/B measurements only: compiled in mpc_b200_drag.cu with the other kernels off the default paths)
    return launch_drag_unit(true, 1, BLOCK, x, u, tf, P, J2, o.kf, o.lin, n_sats, K, 0, o.rtol, o.atol, o.max_step, dst, pitch,
                            offset, status, o.n_nodes, st, DRAG, GENU ? g_ucols : 0);
}

// shipped build (discretize_default_kernel): Phi ping-pongs through the output buffer, 30 KiB of shared memory per warp
std::atomic<int> g_default_block{256};   // mpc_set_tuning(20/21/22): 32 / 128 / 256 threads per CTA

template <bool J2, bool GENU, bool DRAG, int BLOCK>
int launch_default_b(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                     const AdaptiveOpts &o, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status,
                     cudaStream_t st)
{
    if constexpr (DRAG) {
        return launch_drag_unit(true, 0, BLOCK, x, u, tf, P, J2, o.kf, o.lin, n_sats, K, 0, o.rtol, o.atol, o.max_step, dst,
                                pitch, offset, status, o.n_nodes, st);
    } else {
        const size_t smem = (size_t)mpc::kDfSlots * BLOCK * sizeof(double);
        static thread_local int configured_dev = -1;
        const long long n_int = (long long)n_sats * (K - 1);
        const unsigned grid = (unsigned)((n_int + BLOCK - 1) / BLOCK);
        auto kern = mpc::discretize_default_kernel<J2, BLOCK, GENU, false>;
        int rc = configure_smem(kern, smem, configured_dev);
        if (rc) return rc;
        kern<<<grid, BLOCK, smem, st>>>(x, u, tf, P, n_sats, K, g_ucols, o.rtol, o.atol, o.max_step, dst, pitch, offset,
                                        status, o.n_nodes, 0.0, 0.0);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        CUDA_TRY(cudaGetLastError());
        return MPC_SUCCESS;
    }
}

template <bool J2, bool GENU, bool DRAG>
int launch_adaptive_k(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                      const AdaptiveOpts &o, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status,
                      cudaStream_t st)
{
    if (g_default_v1.load(std::memory_order_relaxed))
        return launch_adaptive_v1<J2, GENU, DRAG>(x, u, tf, P, n_sats, K, o, dst, pitch, offset, status, st);
    // The hot loop of this kernel (39 KB of SASS) is larger than the SM's instruction cache.  One-warp CTAs start at
    // different times and walk it out of phase, each paying its own instruction misses (profiles/r02_b: 3.75 warps
    // stalled on instruction fetch per issue).  The warps of ONE large CTA start together and take the same 4-5 steps:
    // they stay within a few cache lines of each other and share every fetched line.  7 warps = 213 KiB of shared memory
    // fill an SM; small batches keep one-warp CTAs so that they still spread over all SMs.  (The drag variant needs 41 KiB
    // per warp: 5 warps.)
    const long long n_int = (long long)n_sats * (K - 1);
    int block = g_default_block.load(std::memory_order_relaxed);
    if (n_int < 148LL * 256) block = 32;
    if (!DRAG) {
        if (block == 256) return launch_default_b<J2, GENU, DRAG, 256>(x, u, tf, P, n_sats, K, o, dst, pitch, offset, status, st);
        if (block == 128 && !GENU) return launch_default_b<J2, GENU, DRAG, 128>(x, u, tf, P, n_sats, K, o, dst, pitch, offset, status, st);
    } else if (block != 32) {
        // the drag branch keeps V_s and a general G_s + W_s as well: 174 slots per thread, 5 warps fill the SM's shared memory
        return launch_default_b<J2, GENU, DRAG, 160>(x, u, tf, P, n_sats, K, o, dst, pitch, offset, status, st);
    }
    return launch_default_b<J2, GENU, DRAG, 32>(x, u, tf, P, n_sats, K, o, dst, pitch, offset, status, st);
}

template <bool J2, bool GENU>
int launch_adaptive_g(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                      const AdaptiveOpts &o, const mpc::DstTab &dst, long long pitch, long long offset, int32_t *status,
                      cudaStream_t st)
{
    if (o.drag) {
        if (GENU) return fail(MPC_E_UNSUPPORTED, "include_drag with u on its own grid is not supported");
        return launch_adaptive_k<J2, false, true>(x, u, tf, P, n_sats, K, o, dst, pitch, offset, status, st);
    }
    return launch_adaptive_k<J2, GENU, false>(x, u, tf, P, n_sats, K, o, dst, pitch, offset, status, st);
}

// The Jacobian's drag terms read const.CD and rho_func / drho_func (linearize_discretize.py:164-169): a constant
// (disc_rho) or the Chebyshev series the host fitted over the radii of the batch (mpc_params::disc_*_cheb).
mpc::DragLin drag_lin(const mpc_params *p)
{
    mpc::DragLin L{};
    L.kc = p->include_drag ? 0.5 * p->disc_cd * p->s_area : 0.0;
    L.n_rho = 1;
    L.rho_c[0] = p->disc_rho;
    if (p->include_drag && p->disc_n_rho > 0) {
        L.r_mid = p->disc_r_mid;
        L.r_ihalf = p->disc_r_ihalf;
        L.n_rho = p->disc_n_rho;
        L.n_drho = p->disc_n_drho;
        for (int i = 0; i < mpc::kRhoCheb; ++i) {
            L.rho_c[i] = i < p->disc_n_rho ? p->disc_rho_cheb[i] : 0.0;
            L.drho_c[i] = i < p->disc_n_drho ? p->disc_drho_cheb[i] : 0.0;
        }
    }
    return L;
}

int check_drag_model(const mpc_params *p)
{
    if (p->include_drag && (p->disc_n_rho < 0 || p->disc_n_rho > MPC_RHO_CHEB || p->disc_n_drho < 0 || p->disc_n_drho > MPC_RHO_CHEB ||
                            (p->disc_n_drho > 0 && p->disc_n_rho == 0) || (p->disc_n_rho > 0 && !(p->disc_r_ihalf > 0.0))))
        return fail(MPC_E_INVALID, "density model of the drag linearisation: need 0 <= disc_n_rho, disc_n_drho <= %d, disc_r_ihalf > 0", MPC_RHO_CHEB);
    return MPC_SUCCESS;
}

void with_drag(AdaptiveOpts &o, const mpc_params *p)
{
    o.drag = p->include_drag;
    o.kf = p->include_drag ? 0.5 * p->c_d * p->s_area * (p->rho_atm / p->rho) : 0.0;
    o.lin = drag_lin(p);
}

int check_adaptive(double rtol, double atol, double max_step)
{
    if (!(rtol > 0.0) || !(atol > 0.0) || !(max_step > 0.0))
        return fail(MPC_E_INVALID, "adaptive mode needs rtol, atol, max_step > 0 (got %g, %g, %g)", rtol, atol, max_step);
    return MPC_SUCCESS;
}

int check_disc_args(const void *x, const void *u, const void *tf, const mpc_params *p, int n_sats, int K, int n_sub)
{
    if (!x || !u || !tf || !p) return fail(MPC_E_INVALID, "null pointer argument");
    if (n_sats < 0 || K < 2 || n_sub < 1)
        return fail(MPC_E_INVALID, "need n_sats >= 0, K >= 2, n_sub >= 1 (got %d, %d, %d)", n_sats, K, n_sub);
    if (p->include_drag && !(p->disc_cd > 0.0 && p->disc_rho >= 0.0))
        // the reference's drag linearisation needs const.CD and a rho_func (linearize_discretize.py:162-169); with
        // its defaults (no CD attribute, rho_func = None) it raises; so do we when they are not supplied
        return fail(MPC_E_UNSUPPORTED, "include_drag needs disc_cd / disc_rho (const.CD, rho_func): the reference raises without them too");
    return check_drag_model(p);
}

// drag branch of the linearisation: coefficients of the dynamics (kf) and of the Jacobian (ka)
double drag_kf(const mpc_params *p) { return 0.5 * p->c_d * p->s_area * (p->rho_atm / p->rho); }

template <bool J2>
int launch_disc_drag(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, double kf, const mpc::DragLin &L,
                     int n_sats, int K, int n_sub, const mpc::DstTab &dst, long long pitch, long long offset,
                     int32_t *status, cudaStream_t st)
{
    mpc::DstTab tab = dst;
    tab.em = em_level();
    return launch_drag_unit(false, 0, 64, x, u, tf, P, J2, kf, L, n_sats, K, n_sub, 0.0, 0.0, 0.0, tab, pitch, offset, status,
                            nullptr, st);
}

// one chunk of a fixed-step discretization on stream st: plain or drag kernel
int launch_fixed(const double *x, const double *u, const double *tf, const mpc_params *p, const mpc::DiscParams &P,
                 int n_sats, int K, int n_sub, const mpc::DstTab &tab, long long pitch, long long offset, int32_t *status,
                 cudaStream_t st)
{
    if (p->include_drag) {
        if (g_ucols > 0) return fail(MPC_E_UNSUPPORTED, "include_drag with u on its own grid is not supported");
        const mpc::DragLin L = drag_lin(p);
        return p->include_j2 ? launch_disc_drag<true>(x, u, tf, P, drag_kf(p), L, n_sats, K, n_sub, tab, pitch, offset, status, st)
                             : launch_disc_drag<false>(x, u, tf, P, drag_kf(p), L, n_sats, K, n_sub, tab, pitch, offset, status, st);
    }
    return p->include_j2 ? launch_disc_n<true, 1>(x, u, tf, P, n_sats, K, n_sub, tab, pitch, offset, status, st)
                         : launch_disc_n<false, 1>(x, u, tf, P, n_sats, K, n_sub, tab, pitch, offset, status, st);
}

int disc_device(const double *x, const double *u, const double *tf, const mpc_params *p, int n_sats, int K,
                int n_sub, double *const *dst, int n_dst, int64_t pitch, int64_t offset, int32_t *status,
                cudaStream_t st)
{
    int rc = check_disc_args(x, u, tf, p, n_sats, K, n_sub);
    if (rc) return rc;
    if (!dst || n_dst < 1 || n_dst > MPC_MAX_DST) return fail(MPC_E_INVALID, "bad destination list");
    const long long n_int = (long long)n_sats * (K - 1);
    if (pitch < offset + n_int || offset < 0) return fail(MPC_E_INVALID, "out_pitch/out_offset do not hold the batch");
    if (n_int == 0) return MPC_SUCCESS;
    mpc::DstTab tab{};
    for (int d = 0; d < mpc::kMaxDst; ++d) tab.p[d] = (d < n_dst) ? dst[d] : nullptr;
    tab.skip_const = g_gather.active ? g_gather.skip_const : g_gather_skip_const.load(std::memory_order_relaxed);
    tab.stagger_phases = g_gather.active ? g_gather.stagger : g_gather_stagger.load(std::memory_order_relaxed);
    tab.km_ntot = g_gather.km_ntot;
    tab.km_soff = g_gather.km_soff;
    if (tab.km_ntot && (p->include_drag || g_ucols > 0 || !g_pair.load(std::memory_order_relaxed)))
        return fail(MPC_E_UNSUPPORTED, "the k-major layout is implemented by the two-node-step kernel only");
    if (tab.stagger_phases > 1) {
        int dev = 0, sms = 148;
        CUDA_TRY(cudaGetDevice(&dev));
        CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        tab.first_wave_ctas = sms * 2;                           // 2 CTAs of 128 threads per SM (launch_disc_n)
        tab.stagger_cycles = (long long)n_sub * 4940LL;          // ~2470 clocks per RK4 step and warp, 2 warps per scheduler
    }
    for (int d = 0; d < n_dst; ++d)
        if (!tab.p[d]) return fail(MPC_E_INVALID, "null destination %d", d);
    const mpc::DiscParams P = disc_params(p);
    if (p->include_drag) {
        if (n_dst != 1) return fail(MPC_E_UNSUPPORTED, "include_drag with several destinations is not supported");
        return launch_fixed(x, u, tf, p, P, n_sats, K, n_sub, tab, pitch, offset, status, st);
    }
    return p->include_j2 ? launch_disc<true>(x, u, tf, P, n_sats, K, n_sub, tab, n_dst, pitch, offset, status, st)
                         : launch_disc<false>(x, u, tf, P, n_sats, K, n_sub, tab, n_dst, pitch, offset, status, st);
}

// ---- ragged batches: satellite s on K_s nodes, buffers padded to Kmax (mpc_discretize_batch_ragged) ----------------------
int check_counts(const int32_t *cnt, int n, int cmax, const char *what)
{
    if (!cnt) return fail(MPC_E_INVALID, "null %s", what);
    for (int s = 0; s < n; ++s)
        if (cnt[s] < 2 || cnt[s] > cmax)
            return fail(MPC_E_INVALID, "%s[%d] = %d: every count must be >= 2 and <= %d", what, s, (int)cnt[s], cmax);
    return MPC_SUCCESS;
}

// first[s] = sum_{r < s} (K_r - 1): the kernels' map from a live interval to (s, k)
std::vector<long long> ragged_first(const int32_t *K_sat, int n)
{
    std::vector<long long> f((size_t)n + 1, 0);
    for (int s = 0; s < n; ++s) f[s + 1] = f[s] + (K_sat[s] - 1);
    return f;
}

// One launch for the batch; the block size follows from the LIVE interval count, as launch_adaptive_k / launch_disc_n
// choose it from n_sats (K-1) for a rectangular batch.  (The thread-group kernel of small rectangular batches has no
// ragged form: small ragged batches take the pair kernel in one-warp CTAs.)
template <bool J2, int BLOCK>
int launch_ragged_default(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                          long long n_live, const long long *first, const AdaptiveOpts &o, const mpc::DstTab &dst,
                          long long pitch, long long offset, int32_t *status, cudaStream_t st)
{
    static thread_local int configured_dev = -1;
    auto kern = mpc::discretize_default_ragged_kernel<J2, BLOCK>;
    const size_t smem = (size_t)mpc::kDfSlots * BLOCK * sizeof(double);
    int rc = configure_smem(kern, smem, configured_dev);
    if (rc) return rc;
    const unsigned grid = (unsigned)((n_live + BLOCK - 1) / BLOCK);
    kern<<<grid, BLOCK, smem, st>>>(x, u, tf, P, n_sats, K, o.rtol, o.atol, o.max_step, dst, pitch, offset, status, o.n_nodes, first);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

template <bool J2, int BLOCK>
int launch_ragged_pair(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                       long long n_live, const long long *first, int n_sub, const mpc::DstTab &dst, long long pitch,
                       long long offset, int32_t *status, cudaStream_t st)
{
    static thread_local int configured_dev = -1;
    auto kern = mpc::discretize_pair_kernel<J2, BLOCK, 255, 1, true>;
    const size_t smem = (size_t)mpc::kDiscSlots * BLOCK * sizeof(double);
    int rc = configure_smem(kern, smem, configured_dev);
    if (rc) return rc;
    const unsigned grid = (unsigned)((n_live + BLOCK - 1) / BLOCK);
    mpc::DstTab tab = dst;
    tab.em = em_level();
    kern<<<grid, BLOCK, smem, st>>>(x, u, tf, P, n_sats, K, n_sub, tab, pitch, offset, status, 0, K - 1, first, nullptr);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

template <bool J2>
int launch_ragged(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                  long long n_live, const long long *first, const AdaptiveOpts *ad, int n_sub, const mpc::DstTab &dst,
                  long long pitch, long long offset, int32_t *status, cudaStream_t st)
{
    if (ad) {
        int block = g_default_block.load(std::memory_order_relaxed);
        if (n_live < 148LL * 256) block = 32;
        if (block == 256) return launch_ragged_default<J2, 256>(x, u, tf, P, n_sats, K, n_live, first, *ad, dst, pitch, offset, status, st);
        if (block == 128) return launch_ragged_default<J2, 128>(x, u, tf, P, n_sats, K, n_live, first, *ad, dst, pitch, offset, status, st);
        return launch_ragged_default<J2, 32>(x, u, tf, P, n_sats, K, n_live, first, *ad, dst, pitch, offset, status, st);
    }
    if (n_live > 148LL * 32 && n_live <= 148LL * 128)
        return launch_ragged_pair<J2, kDiscBlock>(x, u, tf, P, n_sats, K, n_live, first, n_sub, dst, pitch, offset, status, st);
    if (n_live < 148LL * 9 * 32 * 2)
        return launch_ragged_pair<J2, 32>(x, u, tf, P, n_sats, K, n_live, first, n_sub, dst, pitch, offset, status, st);
    return launch_ragged_pair<J2, kDiscBlock>(x, u, tf, P, n_sats, K, n_live, first, n_sub, dst, pitch, offset, status, st);
}

// Per-satellite constants (psc: device DiscParams [n_sats]): one launch for the batch, rectangular (first == nullptr,
// n_units = n_sats (K-1); default mode only) or ragged (n_units live intervals).  The fixed-step form is ragged only: a
// rectangular batch takes it with equal counts, because the rectangular pair kernel with the table spilled where its
// single-constant twin does not (the J2 build: 20 / 56 B against 4 / 40 B), and the ragged one matches its twin.  The block sizes are those launch_disc_n / launch_adaptive_k
// and launch_ragged choose from the same count; the thread-group kernel of small rectangular batches has no such form:
// small batches take the pair kernel in one-warp CTAs, as small ragged batches do.
int launch_units_disc(const double *x, const double *u, const double *tf, const mpc::DiscParams *psc, bool j2, int n_sats,
                      int K, long long n_units, const long long *first, const AdaptiveOpts *ad, int n_sub, const mpc::DstTab &dst,
                      long long pitch, long long offset, int32_t *status, cudaStream_t st)
{
    MpcUnitsDisc a{};
    mpc::DstTab tab = dst;
    tab.em = em_level();
    a.x = x;
    a.u = u;
    a.tf = tf;
    a.psc = psc;
    a.dst_tab = &tab;
    a.first = first;
    a.n_units = n_units;
    a.include_j2 = j2;
    a.n_sats = n_sats;
    a.K = K;
    a.n_sub = n_sub;
    a.adaptive = ad != nullptr;
    if (ad) {
        a.block = g_default_block.load(std::memory_order_relaxed);
        if (n_units < 148LL * 256) a.block = 32;
        a.rtol = ad->rtol;
        a.atol = ad->atol;
        a.max_step = ad->max_step;
        a.n_nodes = ad->n_nodes;
    } else {
        a.block = (n_units > 148LL * 32 && n_units <= 148LL * 128) || n_units >= 148LL * 9 * 32 * 2 ? kDiscBlock : 32;
    }
    a.pitch = pitch;
    a.offset = offset;
    a.status = status;
    a.stream = st;
    CUDA_TRY(mpc_units_launch_disc(&a));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return MPC_SUCCESS;
}

int check_units_disc(const double *x, const double *u, const double *tf, const mpc_params *p, const mpc_sat_consts *consts,
                     int n_sats, int K_max, const int32_t *K_sat, int adaptive, int n_sub, double rtol, double atol, double max_step)
{
    int rc = check_disc_args(x, u, tf, p, n_sats, K_max, adaptive ? 1 : n_sub);
    if (rc) return rc;
    if (p->include_drag) return fail(MPC_E_UNSUPPORTED, "the drag linearisation is not implemented with per-satellite constants");
    if (adaptive && g_default_v1.load(std::memory_order_relaxed))
        return fail(MPC_E_UNSUPPORTED, "the round-1 default-mode kernel (mpc_set_tuning(9)) has no per-satellite-constants form");
    if (adaptive && (rc = check_adaptive(rtol, atol, max_step))) return rc;
    if (K_sat && (rc = check_counts(K_sat, n_sats, K_max, "K_sat"))) return rc;
    return check_sat_consts(consts, n_sats);
}

int check_ragged_disc(const double *x, const double *u, const double *tf, const mpc_params *p, int n_sats, int K_max,
                      const int32_t *K_sat, int adaptive, int n_sub, double rtol, double atol, double max_step)
{
    int rc = check_disc_args(x, u, tf, p, n_sats, K_max, adaptive ? 1 : n_sub);
    if (rc) return rc;
    if (p->include_drag) return fail(MPC_E_UNSUPPORTED, "the drag linearisation is not implemented for ragged batches");
    if (adaptive && (rc = check_adaptive(rtol, atol, max_step))) return rc;
    return check_counts(K_sat, n_sats, K_max, "K_sat");
}

// ---- the default quadrature mode with scipy's RK23 (mpc_discretize_batch_rk23[_host]) ------------------------------------
// consts == nullptr: one constants bag; K_sat == nullptr: a rectangular batch.  The constants are validated as the
// *_units entries validate them; there is no drag branch.
int check_rk23_disc(const double *x, const double *u, const double *tf, const mpc_params *p, const mpc_sat_consts *consts,
                    int n_sats, int K_max, const int32_t *K_sat, double rtol, double atol, double max_step)
{
    int rc = check_disc_args(x, u, tf, p, n_sats, K_max, 1);
    if (rc) return rc;
    if (p->include_drag) return fail(MPC_E_UNSUPPORTED, "the drag linearisation is not implemented with RK23");
    if ((rc = check_adaptive(rtol, atol, max_step))) return rc;
    if (K_sat && (rc = check_counts(K_sat, n_sats, K_max, "K_sat"))) return rc;
    if (consts && (rc = check_sat_consts(consts, n_sats))) return rc;
    if (mpc_rk23_sizeof() != sizeof(mpc::DiscParams)) return fail(MPC_E_CUDA, "mpc_b200_rk23.cu was built against different parameter structs");
    return MPC_SUCCESS;
}

// One launch for the batch (psc: device DiscParams [n_sats] or nullptr; first: device prefix sums or nullptr).  The
// block size follows the default-mode launchers: one-warp CTAs below 148 x 256 threads, full 256-thread CTAs otherwise.
int launch_rk23(const double *x, const double *u, const double *tf, const mpc::DiscParams &P, const mpc::DiscParams *psc,
                bool j2, int n_sats, int K, long long n_units, const long long *first, const AdaptiveOpts &o, double *out,
                long long pitch, long long offset, int32_t *status, cudaStream_t st)
{
    MpcRk23Disc a{};
    a.x = x;
    a.u = u;
    a.tf = tf;
    a.P = &P;
    a.psc = psc;
    a.first = first;
    a.n_units = n_units;
    a.include_j2 = j2;
    a.n_sats = n_sats;
    a.K = K;
    a.block = n_units < 148LL * 256 ? 32 : 256;
    a.rtol = o.rtol;
    a.atol = o.atol;
    a.max_step = o.max_step;
    a.out = out;
    a.pitch = pitch;
    a.offset = offset;
    a.status = status;
    a.n_nodes = o.n_nodes;
    a.stream = st;
    CUDA_TRY(mpc_rk23_launch_disc(&a));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return MPC_SUCCESS;
}

int check_ctrl(const mpc_controller *c)
{
    if (!c) return fail(MPC_E_INVALID, "null controller");
    if (c->kind < MPC_CTRL_ZERO || c->kind > MPC_CTRL_SEQUENCE) return fail(MPC_E_UNSUPPORTED, "unknown controller kind %d", c->kind);
    if (c->kind == MPC_CTRL_SEQUENCE) {
        if (!c->table || c->table_len < 2) return fail(MPC_E_INVALID, "sequence controller needs a table with >= 2 columns");
        if (!c->end_tau_per_sat && !(c->end_tau > 0.0)) return fail(MPC_E_INVALID, "sequence controller needs end_tau > 0");
    }
    return MPC_SUCCESS;
}

// How the propagation is integrated.  n_sub >= 1: fixed-step RK4 with n_sub steps between samples.  n_sub == 0: the
// reference's own integrator (simulator.py:185-187: solve_ivp RK45, max_step = 0.001, scipy's default tolerances, samples
// off the dense output), replayed step for step by propagate_rk45_kernel; `rk` overrides those three numbers.
struct PropMode {
    int n_sub = 0;
    mpc::Rk45Opts rk{1e-3, 1e-6, 1e-3};
    int32_t *n_steps = nullptr;   // RK45 only: steps attempted per satellite (accepted + rejected), may be NULL
    bool rk45() const { return n_sub == 0; }
};

std::atomic<int> g_rk45_spec{1};   // mpc_set_tuning(11/12): speculative first stage of the next step off / on
std::atomic<int> g_rk45_lpw{0};    // mpc_set_tuning(13..16): satellites per warp of the RK45 propagator (0 = automatic)

// satellites per warp: a warp's FP64 instructions cost the same issue slots whether 8 or 32 lanes are active, and the
// propagation is a chain of dependent stages, so a batch is spread over as many SM sub-partitions as there are
// (4 per SM) before warps are filled up
int rk45_lanes_per_warp(int n_sats, int sm_count)
{
    const int forced = g_rk45_lpw.load(std::memory_order_relaxed);
    if (forced > 0) return forced;
    const long long slots = (long long)sm_count * 4;
    for (int lpw = 1; lpw < 32; lpw *= 2)
        if ((long long)n_sats <= slots * lpw) return lpw;
    return 32;
}

template <int KIND, bool DRAG, bool J2>
void launch_rk45(bool overlap, bool spec, unsigned n_warps, cudaStream_t st, const double *y0, const double *tf,
                 const mpc::PropParams &PP, const mpc::CtrlParams &C, const mpc::Rk45Opts &O, int n_sats, int T, int lpw,
                 double *y, double *u_out, int32_t *status, int32_t *n_steps, unsigned int *progress, int seg_len)
{
    // beside the discretization (overlap) the propagation runs as 4-warp CTAs so that it takes CTA slots on few SMs
    if (overlap) {
        const unsigned grid = (n_warps + 3) / 4;
        if (spec)
            mpc::propagate_rk45_kernel<kPropBlockOverlap, KIND, DRAG, J2, true><<<grid, kPropBlockOverlap, 0, st>>>(
                y0, tf, PP, C, O, n_sats, T, lpw, y, u_out, status, n_steps, progress, seg_len);
        else
            mpc::propagate_rk45_kernel<kPropBlockOverlap, KIND, DRAG, J2, false><<<grid, kPropBlockOverlap, 0, st>>>(
                y0, tf, PP, C, O, n_sats, T, lpw, y, u_out, status, n_steps, progress, seg_len);
    } else {
        if (spec)
            mpc::propagate_rk45_kernel<kPropBlock, KIND, DRAG, J2, true><<<n_warps, kPropBlock, 0, st>>>(
                y0, tf, PP, C, O, n_sats, T, lpw, y, u_out, status, n_steps, progress, seg_len);
        else
            mpc::propagate_rk45_kernel<kPropBlock, KIND, DRAG, J2, false><<<n_warps, kPropBlock, 0, st>>>(
                y0, tf, PP, C, O, n_sats, T, lpw, y, u_out, status, n_steps, progress, seg_len);
    }
}

// ragged batch (per-satellite sample counts and / or table lengths): one-warp CTAs, never beside the discretization
template <int KIND, bool DRAG, bool J2>
void launch_rk45_ragged(bool spec, unsigned n_warps, cudaStream_t st, const double *y0, const double *tf, const mpc::PropParams &PP,
                        const mpc::CtrlParams &C, const mpc::Rk45Opts &O, int n_sats, int T, int lpw, double *y, double *u_out,
                        int32_t *status, int32_t *n_steps, const int32_t *T_sat, const int32_t *ku)
{
    if (spec)
        mpc::propagate_rk45_kernel<kPropBlock, KIND, DRAG, J2, true, true><<<n_warps, kPropBlock, 0, st>>>(
            y0, tf, PP, C, O, n_sats, T, lpw, y, u_out, status, n_steps, nullptr, 0, T_sat, ku);
    else
        mpc::propagate_rk45_kernel<kPropBlock, KIND, DRAG, J2, false, true><<<n_warps, kPropBlock, 0, st>>>(
            y0, tf, PP, C, O, n_sats, T, lpw, y, u_out, status, n_steps, nullptr, 0, T_sat, ku);
}

// progress / seg_len: see propagate_kernel (the overlapped pass); then the CTAs are 4 warps instead of 1, so that the
// propagation occupies 32 SMs instead of 128 while the discretization runs beside it.  *progress_target receives the
// value progress[b] reaches when window b may start (warps for the RK4 kernel, satellites for the RK45 one).
int prop_device(const double *y0, const double *tf, const mpc_params *p, const mpc_controller *c,
                const double *table_dev, const double *end_tau_dev, int n_sats, int T, const PropMode &mode, double *y, double *u_out, int32_t *status,
                cudaStream_t st, unsigned int *progress = nullptr, int seg_len = 0, unsigned int *progress_target = nullptr,
                const int32_t *T_sat_dev = nullptr, const int32_t *ku_dev = nullptr, const void *psc_dev = nullptr,
                const mpc::AtmoParams *atmo = nullptr)
{
    // psc_dev: device mpc::PropParams [n_sats] (mpc::AtmoSat [n_sats] with an atmosphere) or NULL
    if (!y0 || !tf || !p || !y) return fail(MPC_E_INVALID, "null pointer argument");
    if (psc_dev && (!mode.rk45() || progress))
        return fail(MPC_E_UNSUPPORTED, "per-satellite constants need the RK45 propagator (n_sub = 0) outside the fused pass");
    if (atmo && (!mode.rk45() || progress))
        return fail(MPC_E_UNSUPPORTED, "an atmosphere needs the RK45 propagator (n_sub = 0) outside the fused pass");
    // per-satellite counts (device arrays here): the RK45 propagator on its own only
    const bool ragged = T_sat_dev || ku_dev;
    if (ragged && (!mode.rk45() || progress))
        return fail(MPC_E_UNSUPPORTED, "per-satellite sample counts / table lengths need the RK45 propagator (n_sub = 0) outside the fused pass");
    const int n_sub = mode.n_sub;
    if (n_sats < 0 || T < 0 || n_sub < 0) return fail(MPC_E_INVALID, "need n_sats >= 0, T >= 0, n_sub >= 0");
    if (mode.rk45() && (!(mode.rk.rtol > 0.0) || !(mode.rk.atol > 0.0) || !(mode.rk.max_step > 0.0)))
        return fail(MPC_E_INVALID, "the RK45 propagator needs rtol, atol, max_step > 0");
    int rc = check_ctrl(c);
    if (rc) return rc;
    if (n_sats == 0 || T == 0) return MPC_SUCCESS;
    mpc::CtrlParams C;
    C.kind = c->kind;
    C.table_len = c->table_len;
    C.table_per_sat = c->table_per_sat;
    C.pad = 0;
    C.t0 = c->thrust[0];
    C.t1 = c->thrust[1];
    C.t2 = c->thrust[2];
    C.end_tau = c->end_tau;
    C.table = (c->kind == MPC_CTRL_SEQUENCE) ? table_dev : nullptr;
    C.end_tau_arr = (c->kind == MPC_CTRL_SEQUENCE) ? end_tau_dev : nullptr;
    if (c->kind != MPC_CTRL_SEQUENCE) ku_dev = nullptr;
    const unsigned grid = (unsigned)((n_sats + kPropBlock - 1) / kPropBlock);
    const unsigned grid_ov = (unsigned)((n_sats + kPropBlockOverlap - 1) / kPropBlockOverlap);
    const mpc::PropParams PP = atmo ? atmo_prop_params(p) : prop_params(p);
    int dev = 0, sms = 148;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    // beside the discretization full warps keep the propagation on few SMs; on its own it spreads out
    const int lpw = progress ? 32 : rk45_lanes_per_warp(n_sats, sms);
    const unsigned n_warps = (unsigned)((n_sats + lpw - 1) / lpw);
    const bool spec = g_rk45_spec.load(std::memory_order_relaxed) != 0;
    if (progress_target) *progress_target = mode.rk45() ? (unsigned)n_sats : (unsigned)((n_sats + 31) / 32);
    if (psc_dev || atmo) {   // per-satellite constants / the atmosphere: one-warp CTAs, mpc_b200_units.cu / mpc_b200_atmo.cu
        MpcUnitsProp a{};
        a.y0 = y0;
        a.tf = tf;
        a.psc = psc_dev;
        a.ctrl = &C;
        a.opts = &mode.rk;
        a.kind = c->kind;
        a.include_drag = p->include_drag;
        a.include_j2 = p->include_j2;
        a.n_sats = n_sats;
        a.T = T;
        a.lpw = lpw;
        a.n_warps = n_warps;
        a.y = y;
        a.u_out = u_out;
        a.status = status;
        a.n_steps = mode.n_steps;
        a.T_sat = T_sat_dev;
        a.ku = ku_dev;
        a.stream = st;
        a.prop = &PP;
        if (atmo) CUDA_TRY(mpc_atmo_launch_rk45(&a, atmo));
        else CUDA_TRY(mpc_units_launch_rk45(&a));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return MPC_SUCCESS;
    }
    // one straight-line kernel per (controller law, drag, J2)
#define MPC_PROP(KIND, DRAG, J2)                                                                                          \
    do {                                                                                                                  \
        if (ragged)                                                                                                       \
            launch_rk45_ragged<KIND, DRAG, J2>(spec, n_warps, st, y0, tf, PP, C, mode.rk, n_sats, T, lpw, y, u_out, status,  \
                                               mode.n_steps, T_sat_dev, ku_dev);                                           \
        else if (mode.rk45())                                                                                             \
            launch_rk45<KIND, DRAG, J2>(progress != nullptr, spec, n_warps, st, y0, tf, PP, C, mode.rk, n_sats, T, lpw, y, \
                                        u_out, status, mode.n_steps, progress, seg_len);                                  \
        else if (progress)                                                                                                \
            mpc::propagate_kernel<kPropBlockOverlap, KIND, DRAG, J2><<<grid_ov, kPropBlockOverlap, 0, st>>>(              \
                y0, tf, PP, C, n_sats, T, n_sub, y, u_out, status, progress, seg_len);                                    \
        else                                                                                                              \
            mpc::propagate_kernel<kPropBlock, KIND, DRAG, J2><<<grid, kPropBlock, 0, st>>>(y0, tf, PP, C, n_sats, T,      \
                                                                                           n_sub, y, u_out, status);     \
    } while (0)
#define MPC_PROP_K(KIND)                                   \
    do {                                                   \
        if (p->include_drag) {                             \
            if (p->include_j2) MPC_PROP(KIND, true, true); \
            else MPC_PROP(KIND, true, false);              \
        } else {                                           \
            if (p->include_j2) MPC_PROP(KIND, false, true); \
            else MPC_PROP(KIND, false, false);             \
        }                                                  \
    } while (0)
    switch (c->kind) {
        case MPC_CTRL_ZERO: MPC_PROP_K(0); break;
        case MPC_CTRL_CONSTANT: MPC_PROP_K(1); break;
        case MPC_CTRL_TANGENTIAL: MPC_PROP_K(2); break;
        default: MPC_PROP_K(3); break;
    }
#undef MPC_PROP_K
#undef MPC_PROP
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

PropMode mode_of(int n_sub)
{
    PropMode m;
    m.n_sub = n_sub;
    return m;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
struct mpc_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t s_compute = nullptr, s_copy = nullptr;
    std::vector<cudaEvent_t> ev;  // one per chunk slot
    // grow-only device workspace
    double *d_x = nullptr, *d_u = nullptr, *d_tf = nullptr, *d_out = nullptr, *d_y0 = nullptr, *d_tab = nullptr;
    int32_t *d_status = nullptr, *d_status2 = nullptr, *d_nodes = nullptr;
    double *d_endtau = nullptr;
    long long *d_first = nullptr;            // ragged batches: prefix sums of K_s - 1
    int32_t *d_cnt = nullptr;                // ragged batches: T_sat and table_len_sat
    size_t cap_first = 0, cap_cnt = 0;
    double *d_psc = nullptr;                 // per-satellite constants: the derived kernel constants (*_units_host)
    size_t cap_psc = 0;
    double *d_conj = nullptr;                // conjunction screening (mpc_screen_conjunctions_host): scratch, events,
    double *d_conj_ev = nullptr;             // counters
    unsigned long long *d_conj_cnt = nullptr;
    size_t cap_conj = 0, cap_conj_ev = 0, cap_conj_cnt = 0;
    cudaStream_t s_pushk = nullptr;          // high-priority stream of the copy kernels (push gather, SM-driven variant)
    cudaStream_t s_aux[3] = {};              // compute streams the chunk kernels of the push gather rotate over
    cudaStream_t s_push[MPC_MAX_DST] = {};   // one stream per peer for the copy-engine gather (mpc_discretize_batch_push)
    std::vector<cudaEvent_t> ev_push;       // [chunk] kernel-done events + [MPC_MAX_DST] stream-join events
    // overlapped propagate -> discretize pass (mpc_propagate_discretize)
    cudaStream_t s_prop = nullptr, s_win[2] = {};   // propagation (highest priority) / discretization windows
    cudaEvent_t ev_ov[4] = {};                      // fork + three joins
    unsigned int *d_progress = nullptr;             // [kMaxWindows] warps of the propagation past each window's last sample
    int32_t *h_stage = nullptr;  // pinned staging for the int32 status / node-count words (caller buffers may be pageable)
    size_t cap_stage = 0;
    size_t cap_nodes = 0, cap_endtau = 0;
    size_t cap_x = 0, cap_u = 0, cap_tf = 0, cap_out = 0, cap_y0 = 0, cap_tab = 0, cap_status = 0, cap_status2 = 0;
};

namespace {

template <typename T>
int ensure(T *&ptr, size_t &cap, size_t count)
{
    if (count <= cap) return MPC_SUCCESS;
    if (ptr) CUDA_TRY(cudaFree(ptr));
    ptr = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc((void **)&ptr, count * sizeof(T));
    if (e != cudaSuccess) return fail(MPC_E_NOMEM, "cudaMalloc of %zu bytes failed: %s", count * sizeof(T), cudaGetErrorString(e));
    cap = count;
    return MPC_SUCCESS;
}

int ensure_stage(mpc_ctx *ctx, size_t count)
{
    if (count <= ctx->cap_stage) return MPC_SUCCESS;
    if (ctx->h_stage) CUDA_TRY(cudaFreeHost(ctx->h_stage));
    ctx->h_stage = nullptr;
    ctx->cap_stage = 0;
    if (cudaHostAlloc((void **)&ctx->h_stage, count * sizeof(int32_t), cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return fail(MPC_E_NOMEM, "cudaHostAlloc of %zu bytes failed", count * sizeof(int32_t));
    }
    ctx->cap_stage = count;
    return MPC_SUCCESS;
}

// true when p is page-locked host memory (mpc_host_alloc / cudaHostAlloc / cudaHostRegister): an async copy into it
// does not block the enqueuing thread, so no staging is needed
bool is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

int ensure_events(mpc_ctx *ctx, size_t n)
{
    while (ctx->ev.size() < n) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->ev.push_back(e);
    }
    return MPC_SUCCESS;
}

// Satellites per chunk of the host pipeline: one wave of the discretization kernel (9 one-warp CTAs per SM in
// the small-batch configuration launch_disc_n picks for a chunk of this size), so that no chunk ends in a
// partially filled wave, the first D2H starts after ~0.3 ms and the copy engine then never idles.
int chunk_sats(const mpc_ctx *ctx, int n_sats, int K)
{
    const long long per_sat = std::max(1, K - 1);
    const long long wave = (long long)ctx->sm_count * 9 * 32;
    return (int)std::min<long long>(std::max<long long>(wave / per_sat, 1), std::max(n_sats, 1));
}

// Rows 42..48 of the SoA result are the last row of A_k = Phi(tau_{k+1}).  The last row of the Jacobian A is
// zero (linearize_discretize.py:177-179), so that row of Phi never leaves its initial value e7^T: the kernels
// store the constants 0,0,0,0,0,0,1 there.  The host pipeline does not move 7/105 of the result over PCIe for
// that: it copies rows [0,42) and [49,105) and writes the seven constant rows into the host buffer itself
// while the DMA engine is busy.
constexpr int kConstRow0 = MPC_ROW_A + 42, kConstRow1 = MPC_ROW_A + 49;

// D2H of the columns [c0, c0+nc) of the SoA result (all rows but the constant ones), host pitch = n_int
int copy_out_chunk(double *out_host, const double *d_out, long long n_int, long long c0, long long nc, cudaStream_t st)
{
    const size_t pitch = (size_t)n_int * sizeof(double), width = (size_t)nc * sizeof(double);
    CUDA_TRY(cudaMemcpy2DAsync(out_host + c0, pitch, d_out + c0, pitch, width, kConstRow0, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpy2DAsync(out_host + (size_t)kConstRow1 * n_int + c0, pitch, d_out + (size_t)kConstRow1 * n_int + c0,
                               pitch, width, MPC_OUT_ROWS - kConstRow1, cudaMemcpyDeviceToHost, st));
    return MPC_SUCCESS;
}

void fill_const_rows(double *out_host, long long n_int)
{
    memset(out_host + (size_t)kConstRow0 * n_int, 0, (size_t)6 * n_int * sizeof(double));
    double *one = out_host + (size_t)(kConstRow1 - 1) * n_int;
    for (long long i = 0; i < n_int; ++i) one[i] = 1.0;
}

}  // namespace

extern "C" {

int mpc_version(void) { return MPC_B200_VERSION; }

const char *mpc_last_error(void) { return g_err; }

int mpc_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int mpc_device_info(int device, char *name, int name_len, int *sm_count, int *cc_major, int *cc_minor)
{
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (name && name_len > 0) {
        strncpy(name, prop.name, (size_t)name_len - 1);
        name[name_len - 1] = 0;
    }
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return MPC_SUCCESS;
}

int64_t mpc_launch_count(void) { return (int64_t)g_launches.load(); }

int mpc_set_gather_tuning(int skip_const, int stagger_phases)
{
    if (skip_const < 0 || skip_const > 2 || stagger_phases < 0 || stagger_phases > 64)
        return fail(MPC_E_INVALID, "bad gather tuning (%d, %d)", skip_const, stagger_phases);
    g_gather_skip_const.store(skip_const);
    g_gather_stagger.store(stagger_phases);
    return MPC_SUCCESS;
}

int mpc_set_tuning(int variant)
{
    if (variant == 7 || variant == 8) {   // 7: one integrator step per node everywhere; 8: two-node steps back on
        g_pair.store(variant == 8);
        return MPC_SUCCESS;
    }
    if (variant == 9 || variant == 10) {  // 9: round-1 build of the default-mode kernel; 10: back to the shipped one
        g_default_v1.store(variant == 9);
        return MPC_SUCCESS;
    }
    if (variant == 11 || variant == 12) {  // RK45 propagator: speculative first stage of the next step off / on
        g_rk45_spec.store(variant == 12);
        return MPC_SUCCESS;
    }
    if (variant >= 13 && variant <= 19) {  // RK45 propagator: satellites per warp 13 automatic, 14..19 -> 32,16,8,4,2,1
        static const int lpw[7] = {0, 32, 16, 8, 4, 2, 1};
        g_rk45_lpw.store(lpw[variant - 13]);
        return MPC_SUCCESS;
    }
    if (variant >= 26 && variant <= 29) {  // streamed host pass (k-major): number of k-windows
        g_host_windows.store(16 * (variant - 25));
        return MPC_SUCCESS;
    }
    if (variant >= 23 && variant <= 25) {  // small batches: 8-lanes-per-interval kernel off / on / at any size
        g_group.store(variant - 23);
        return MPC_SUCCESS;
    }
    if (variant == 37 || variant == 38) {  // 101-node trapezoid sums through their Euler-Maclaurin expansion: off / on
        g_em.store(variant - 37);
        return MPC_SUCCESS;
    }
    if (variant == 39 || variant == 40) {  // 11-node form of the 101-node sums on fifth-order steps: off / on
        g_em3.store(variant - 39);
        return MPC_SUCCESS;
    }
    if (variant >= 20 && variant <= 22) {  // default-mode kernel: threads per CTA 32 / 128 / 256
        static const int blk[3] = {32, 128, 256};
        g_default_block.store(blk[variant - 20]);
        return MPC_SUCCESS;
    }
    if (variant < 0 || variant > 6) return fail(MPC_E_INVALID, "unknown tuning variant %d", variant);
    g_tuning.store(variant);
    return MPC_SUCCESS;
}

int mpc_discretize_batch(const double *x, const double *u, const double *tf, const mpc_params *p, int n_sats,
                         int K, int n_sub, double *out, int64_t out_pitch, int64_t out_offset, int32_t *status,
                         void *stream)
{
    double *dst[1] = {out};
    return disc_device(x, u, tf, p, n_sats, K, n_sub, dst, 1, out_pitch, out_offset, status, (cudaStream_t)stream);
}

int mpc_discretize_batch_multi(const double *x, const double *u, const double *tf, const mpc_params *p,
                               int n_sats, int K, int n_sub, double *const *dst, int n_dst, int64_t out_pitch,
                               int64_t out_offset, int32_t *status, void *stream)
{
    return disc_device(x, u, tf, p, n_sats, K, n_sub, dst, n_dst, out_pitch, out_offset, status,
                       (cudaStream_t)stream);
}

int mpc_discretize_batch_adaptive(const double *x, const double *u, const double *tf, const mpc_params *p,
                                  int n_sats, int K, double rtol, double atol, double max_step, double *out,
                                  int64_t out_pitch, int64_t out_offset, int32_t *status, int32_t *n_nodes, void *stream)
{
    int rc = check_disc_args(x, u, tf, p, n_sats, K, 1);
    if (rc) return rc;
    if ((rc = check_adaptive(rtol, atol, max_step))) return rc;
    if (!out) return fail(MPC_E_INVALID, "null output");
    const long long n_int = (long long)n_sats * (K - 1);
    if (out_pitch < out_offset + n_int || out_offset < 0) return fail(MPC_E_INVALID, "out_pitch/out_offset do not hold the batch");
    if (n_int == 0) return MPC_SUCCESS;
    mpc::DstTab tab{};
    tab.p[0] = out;
    AdaptiveOpts o{rtol, atol, max_step, n_nodes};
    with_drag(o, p);
    const mpc::DiscParams P = disc_params(p);
    return p->include_j2 ? launch_adaptive<true>(x, u, tf, P, n_sats, K, o, tab, out_pitch, out_offset, status, (cudaStream_t)stream)
                         : launch_adaptive<false>(x, u, tf, P, n_sats, K, o, tab, out_pitch, out_offset, status, (cudaStream_t)stream);
}

int mpc_discretize_batch_ugrid(const double *x, const double *u, int u_cols, const double *tf, const mpc_params *p,
                               int n_sats, int K, int adaptive, int n_sub, double rtol, double atol, double max_step,
                               double *out, int64_t out_pitch, int64_t out_offset, int32_t *status, int32_t *n_nodes,
                               void *stream)
{
    if (u_cols < 2) return fail(MPC_E_INVALID, "u needs at least 2 columns (got %d)", u_cols);
    UcolsScope scope(u_cols);
    if (adaptive)
        return mpc_discretize_batch_adaptive(x, u, tf, p, n_sats, K, rtol, atol, max_step, out, out_pitch, out_offset,
                                             status, n_nodes, stream);
    return mpc_discretize_batch(x, u, tf, p, n_sats, K, n_sub, out, out_pitch, out_offset, status, stream);
}

int mpc_discretize_batch_ragged(const double *x, const double *u, const double *tf, const mpc_params *p, int n_sats,
                                int K_max, const int32_t *K_sat, int64_t *first, int adaptive, int n_sub, double rtol,
                                double atol, double max_step, double *out, int64_t out_pitch, int64_t out_offset,
                                int32_t *status, int32_t *n_nodes, void *stream)
{
    int rc = check_ragged_disc(x, u, tf, p, n_sats, K_max, K_sat, adaptive, n_sub, rtol, atol, max_step);
    if (rc) return rc;
    if (!out || !first) return fail(MPC_E_INVALID, "null output / first");
    if (out_pitch < out_offset + (long long)n_sats * (K_max - 1) || out_offset < 0)
        return fail(MPC_E_INVALID, "out_pitch/out_offset do not hold the batch");
    if (n_sats == 0) return MPC_SUCCESS;
    cudaStream_t st = (cudaStream_t)stream;
    const std::vector<long long> f = ragged_first(K_sat, n_sats);
    // (pageable source: cudaMemcpyAsync stages it before returning, the vector may go)
    CUDA_TRY(cudaMemcpyAsync(first, f.data(), f.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    mpc::DstTab tab{};
    tab.p[0] = out;
    const AdaptiveOpts o{rtol, atol, max_step, n_nodes};
    const mpc::DiscParams P = disc_params(p);
    const long long *fd = (const long long *)first;
    return p->include_j2 ? launch_ragged<true>(x, u, tf, P, n_sats, K_max, f[n_sats], fd, adaptive ? &o : nullptr, n_sub, tab, out_pitch, out_offset, status, st)
                         : launch_ragged<false>(x, u, tf, P, n_sats, K_max, f[n_sats], fd, adaptive ? &o : nullptr, n_sub, tab, out_pitch, out_offset, status, st);
}

int mpc_propagate_batch(const double *y0, const double *tf, const mpc_params *p, const mpc_controller *ctrl,
                        int n_sats, int T, int n_sub, double *y, double *u_out, int32_t *status, void *stream)
{
    return prop_device(y0, tf, p, ctrl, ctrl ? ctrl->table : nullptr, ctrl ? ctrl->end_tau_per_sat : nullptr, n_sats, T,
                       mode_of(n_sub), y, u_out, status,
                       (cudaStream_t)stream);
}

int mpc_propagate_batch_rk45(const double *y0, const double *tf, const mpc_params *p, const mpc_controller *ctrl,
                             int n_sats, int T, double rtol, double atol, double max_step, double *y, double *u_out,
                             int32_t *status, int32_t *n_steps, void *stream)
{
    PropMode m;
    m.rk = mpc::Rk45Opts{rtol, atol, max_step};
    m.n_steps = n_steps;
    return prop_device(y0, tf, p, ctrl, ctrl ? ctrl->table : nullptr, ctrl ? ctrl->end_tau_per_sat : nullptr, n_sats, T, m,
                       y, u_out, status, (cudaStream_t)stream);
}

int mpc_propagate_batch_rk45_ragged(const double *y0, const double *tf, const mpc_params *p, const mpc_controller *ctrl,
                                    int n_sats, int T_max, const int32_t *T_sat, const int32_t *table_len_sat, double rtol,
                                    double atol, double max_step, double *y, double *u_out, int32_t *status,
                                    int32_t *n_steps, void *stream)
{
    if (!T_sat) return fail(MPC_E_INVALID, "null T_sat");
    if (T_max < 2) return fail(MPC_E_INVALID, "need T_max >= 2 (got %d)", T_max);
    PropMode m;
    m.rk = mpc::Rk45Opts{rtol, atol, max_step};
    m.n_steps = n_steps;
    return prop_device(y0, tf, p, ctrl, ctrl ? ctrl->table : nullptr, ctrl ? ctrl->end_tau_per_sat : nullptr, n_sats, T_max, m,
                       y, u_out, status, (cudaStream_t)stream, nullptr, 0, nullptr, T_sat, table_len_sat);
}

int mpc_ctx_create(int device, mpc_ctx **out)
{
    if (!out) return fail(MPC_E_INVALID, "null ctx pointer");
    int n = 0;
    CUDA_TRY(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(MPC_E_INVALID, "device %d out of range (%d visible)", device, n);
    CUDA_TRY(cudaSetDevice(device));
    mpc_ctx *c = new mpc_ctx();
    c->device = device;
    CUDA_TRY(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
    CUDA_TRY(cudaStreamCreateWithFlags(&c->s_compute, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&c->s_copy, cudaStreamNonBlocking));
    *out = c;
    return MPC_SUCCESS;
}

int mpc_ctx_destroy(mpc_ctx *c)
{
    if (!c) return MPC_SUCCESS;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (cudaEvent_t e : c->ev) cudaEventDestroy(e);
    if (c->s_compute) cudaStreamDestroy(c->s_compute);
    if (c->s_copy) cudaStreamDestroy(c->s_copy);
    for (cudaStream_t ps : c->s_push)
        if (ps) cudaStreamDestroy(ps);
    for (cudaStream_t ps : c->s_aux)
        if (ps) cudaStreamDestroy(ps);
    if (c->s_pushk) cudaStreamDestroy(c->s_pushk);
    if (c->s_prop) cudaStreamDestroy(c->s_prop);
    for (cudaStream_t w : c->s_win)
        if (w) cudaStreamDestroy(w);
    for (cudaEvent_t e : c->ev_ov)
        if (e) cudaEventDestroy(e);
    cudaFree(c->d_progress);
    for (cudaEvent_t e : c->ev_push) cudaEventDestroy(e);
    cudaFree(c->d_x);
    cudaFree(c->d_u);
    cudaFree(c->d_tf);
    cudaFree(c->d_out);
    cudaFree(c->d_y0);
    cudaFree(c->d_tab);
    cudaFree(c->d_status);
    cudaFree(c->d_status2);
    cudaFree(c->d_nodes);
    cudaFree(c->d_endtau);
    cudaFree(c->d_first);
    cudaFree(c->d_cnt);
    cudaFree(c->d_psc);
    cudaFree(c->d_conj);
    cudaFree(c->d_conj_ev);
    cudaFree(c->d_conj_cnt);
    if (c->h_stage) cudaFreeHost(c->h_stage);
    delete c;
    return MPC_SUCCESS;
}

void *mpc_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        fail(MPC_E_NOMEM, "cudaHostAlloc of %zu bytes failed", bytes);
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void mpc_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

// shared body of the two host-buffer discretization entry points (ad == nullptr: fixed-step kernel)
// K_sat != nullptr: a ragged batch (K = Kmax, mpc_discretize_batch_ragged_host)
// consts != nullptr: per-satellite constants (mpc_discretize_batch_units_host), rectangular or ragged
static int disc_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf, const mpc_params *p, int n_sats,
                     int K, int n_sub, const AdaptiveOpts *ad, double *out_host, int32_t *status_host,
                     int32_t *n_nodes_host, const int32_t *K_sat = nullptr, const mpc_sat_consts *consts = nullptr)
{
    if (!ctx || !out_host) return fail(MPC_E_INVALID, "null ctx/out");
    const bool rk23 = ad && ad->rk23;
    int rc = rk23 ? check_rk23_disc(x, u, tf, p, consts, n_sats, K, K_sat, ad->rtol, ad->atol, ad->max_step)
           : consts ? check_units_disc(x, u, tf, p, consts, n_sats, K, K_sat, ad != nullptr, n_sub, ad ? ad->rtol : 0.0,
                                       ad ? ad->atol : 0.0, ad ? ad->max_step : 0.0)
           : K_sat ? check_ragged_disc(x, u, tf, p, n_sats, K, K_sat, ad != nullptr, n_sub, ad ? ad->rtol : 0.0, ad ? ad->atol : 0.0,
                                       ad ? ad->max_step : 0.0)
                   : check_disc_args(x, u, tf, p, n_sats, K, n_sub);
    if (rc) return rc;
    if (ad && (rc = check_adaptive(ad->rtol, ad->atol, ad->max_step))) return rc;
    const long long n_int = (long long)n_sats * (K - 1);
    if (n_int == 0) return MPC_SUCCESS;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if ((rc = ensure(ctx->d_x, ctx->cap_x, (size_t)n_sats * 7 * K))) return rc;
    const int Ku = g_ucols > 0 ? g_ucols : K;   // columns of u (its own grid in the *_ugrid entry points)
    if ((rc = ensure(ctx->d_u, ctx->cap_u, (size_t)n_sats * 3 * Ku))) return rc;
    if ((rc = ensure(ctx->d_tf, ctx->cap_tf, (size_t)n_sats))) return rc;
    if ((rc = ensure(ctx->d_out, ctx->cap_out, (size_t)n_int * MPC_OUT_ROWS))) return rc;
    if ((rc = ensure(ctx->d_status, ctx->cap_status, (size_t)n_int))) return rc;
    if (ad && n_nodes_host && (rc = ensure(ctx->d_nodes, ctx->cap_nodes, (size_t)n_int))) return rc;
    const int cs = chunk_sats(ctx, n_sats, K);
    const int n_chunks = (n_sats + cs - 1) / cs;
    if ((rc = ensure_events(ctx, (size_t)n_chunks))) return rc;
    const mpc::DiscParams P = disc_params(p);
    CUDA_TRY(cudaMemcpyAsync(ctx->d_tf, tf, (size_t)n_sats * sizeof(double), cudaMemcpyHostToDevice, ctx->s_compute));
    std::vector<long long> first;
    if (K_sat) {
        first = ragged_first(K_sat, n_sats);
        if ((rc = ensure(ctx->d_first, ctx->cap_first, first.size()))) return rc;
        CUDA_TRY(cudaMemcpyAsync(ctx->d_first, first.data(), first.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->s_compute));
    }
    if (consts) {
        if ((rc = ensure(ctx->d_psc, ctx->cap_psc, (size_t)n_sats * MPC_SAT_SCRATCH_DOUBLES))) return rc;
        if ((rc = upload_sat_table<mpc::DiscParams>(p, consts, n_sats, ctx->d_psc, ctx->s_compute, disc_params))) return rc;
    }
    const mpc::DiscParams *psc = (const mpc::DiscParams *)ctx->d_psc;
    for (int c = 0; c < n_chunks; ++c) {
        const int s0 = c * cs, ns = std::min(cs, n_sats - s0);
        const double *dx = ctx->d_x + (size_t)s0 * 7 * K, *du = ctx->d_u + (size_t)s0 * 3 * Ku;
        CUDA_TRY(cudaMemcpyAsync((void *)dx, x + (size_t)s0 * 7 * K, (size_t)ns * 7 * K * sizeof(double),
                                 cudaMemcpyHostToDevice, ctx->s_compute));
        CUDA_TRY(cudaMemcpyAsync((void *)du, u + (size_t)s0 * 3 * Ku, (size_t)ns * 3 * Ku * sizeof(double),
                                 cudaMemcpyHostToDevice, ctx->s_compute));
        mpc::DstTab tab{};
        tab.p[0] = ctx->d_out;
        const long long off = (long long)s0 * (K - 1);
        if (rk23) {
            AdaptiveOpts o = *ad;
            o.n_nodes = n_nodes_host ? ctx->d_nodes + off : nullptr;
            long long n_units = (long long)ns * (K - 1);
            if (K_sat) {   // the padding columns as in the ragged branch below
                CUDA_TRY(cudaMemset2DAsync(ctx->d_out + off, (size_t)n_int * sizeof(double), 0xFF, (size_t)n_units * sizeof(double),
                                           MPC_OUT_ROWS, ctx->s_compute));
                CUDA_TRY(cudaMemsetAsync(ctx->d_status + off, 0, (size_t)n_units * sizeof(int32_t), ctx->s_compute));
                if (n_nodes_host) CUDA_TRY(cudaMemsetAsync(ctx->d_nodes + off, 0, (size_t)n_units * sizeof(int32_t), ctx->s_compute));
                n_units = first[s0 + ns] - first[s0];
            }
            rc = launch_rk23(dx, du, ctx->d_tf + s0, P, consts ? psc + s0 : nullptr, p->include_j2, ns, K, n_units,
                             K_sat ? ctx->d_first + s0 : nullptr, o, ctx->d_out, n_int, off, ctx->d_status + off, ctx->s_compute);
        } else if (consts && !K_sat) {
            AdaptiveOpts o = ad ? *ad : AdaptiveOpts{};
            o.n_nodes = (ad && n_nodes_host) ? ctx->d_nodes + off : nullptr;
            rc = launch_units_disc(dx, du, ctx->d_tf + s0, psc + s0, p->include_j2, ns, K, (long long)ns * (K - 1), nullptr,
                                   ad ? &o : nullptr, n_sub, tab, n_int, off, ctx->d_status + off, ctx->s_compute);
        } else if (K_sat) {
            // the kernel leaves the padding columns alone: they go back as NaN (all-ones bytes) / status 0 / 0 nodes
            const long long nc = (long long)ns * (K - 1);
            CUDA_TRY(cudaMemset2DAsync(ctx->d_out + off, (size_t)n_int * sizeof(double), 0xFF, (size_t)nc * sizeof(double),
                                       MPC_OUT_ROWS, ctx->s_compute));
            CUDA_TRY(cudaMemsetAsync(ctx->d_status + off, 0, (size_t)nc * sizeof(int32_t), ctx->s_compute));
            if (ad && n_nodes_host) CUDA_TRY(cudaMemsetAsync(ctx->d_nodes + off, 0, (size_t)nc * sizeof(int32_t), ctx->s_compute));
            AdaptiveOpts o = ad ? *ad : AdaptiveOpts{};
            o.n_nodes = (ad && n_nodes_host) ? ctx->d_nodes + off : nullptr;
            if (consts)
                rc = launch_units_disc(dx, du, ctx->d_tf + s0, psc + s0, p->include_j2, ns, K, first[s0 + ns] - first[s0],
                                       ctx->d_first + s0, ad ? &o : nullptr, n_sub, tab, n_int, off, ctx->d_status + off, ctx->s_compute);
            else
                rc = p->include_j2 ? launch_ragged<true>(dx, du, ctx->d_tf + s0, P, ns, K, first[s0 + ns] - first[s0], ctx->d_first + s0,
                                                         ad ? &o : nullptr, n_sub, tab, n_int, off, ctx->d_status + off, ctx->s_compute)
                                   : launch_ragged<false>(dx, du, ctx->d_tf + s0, P, ns, K, first[s0 + ns] - first[s0], ctx->d_first + s0,
                                                          ad ? &o : nullptr, n_sub, tab, n_int, off, ctx->d_status + off, ctx->s_compute);
        } else if (ad) {
            AdaptiveOpts o = *ad;
            with_drag(o, p);
            o.n_nodes = n_nodes_host ? ctx->d_nodes + off : nullptr;
            rc = p->include_j2 ? launch_adaptive<true>(dx, du, ctx->d_tf + s0, P, ns, K, o, tab, n_int, off, ctx->d_status + off, ctx->s_compute)
                               : launch_adaptive<false>(dx, du, ctx->d_tf + s0, P, ns, K, o, tab, n_int, off, ctx->d_status + off, ctx->s_compute);
        } else {
            rc = launch_fixed(dx, du, ctx->d_tf + s0, p, P, ns, K, n_sub, tab, n_int, off, ctx->d_status + off, ctx->s_compute);
        }
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(ctx->ev[c], ctx->s_compute));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_copy, ctx->ev[c], 0));
        if ((rc = copy_out_chunk(out_host, ctx->d_out, n_int, off, (long long)ns * (K - 1), ctx->s_copy))) return rc;
    }
    // The host writes the structural constants while the GPU / DMA engine work.  The int32 words go through
    // pinned staging: a copy into a pageable caller buffer would block this thread until the whole pipeline drains.
    fill_const_rows(out_host, n_int);
    if (K_sat) {   // ... but not in the padding columns of a ragged batch
        const double qnan = std::numeric_limits<double>::quiet_NaN();
        for (int r = kConstRow0; r < kConstRow1; ++r)
            for (int sv = 0; sv < n_sats; ++sv)
                for (long long k = K_sat[sv] - 1; k < K - 1; ++k) out_host[(size_t)r * n_int + (size_t)sv * (K - 1) + k] = qnan;
    }
    const bool want_nodes = ad && n_nodes_host;
    if ((rc = ensure_stage(ctx, (size_t)n_int * 2))) return rc;
    int32_t *st_dst = status_host ? (is_pinned(status_host) ? status_host : ctx->h_stage) : nullptr;
    int32_t *nn_dst = want_nodes ? (is_pinned(n_nodes_host) ? n_nodes_host : ctx->h_stage + n_int) : nullptr;
    if (st_dst)
        CUDA_TRY(cudaMemcpyAsync(st_dst, ctx->d_status, (size_t)n_int * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->s_copy));
    if (nn_dst)
        CUDA_TRY(cudaMemcpyAsync(nn_dst, ctx->d_nodes, (size_t)n_int * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->s_copy));
    CUDA_TRY(cudaStreamSynchronize(ctx->s_copy));
    CUDA_TRY(cudaStreamSynchronize(ctx->s_compute));
    if (st_dst && st_dst != status_host) memcpy(status_host, st_dst, (size_t)n_int * sizeof(int32_t));
    if (nn_dst && nn_dst != n_nodes_host) memcpy(n_nodes_host, nn_dst, (size_t)n_int * sizeof(int32_t));
    return MPC_SUCCESS;
}

int mpc_discretize_batch_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf,
                              const mpc_params *p, int n_sats, int K, int n_sub, double *out_host,
                              int32_t *status_host)
{
    return disc_host(ctx, x, u, tf, p, n_sats, K, n_sub, nullptr, out_host, status_host, nullptr);
}

int mpc_discretize_batch_ragged_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf, const mpc_params *p,
                                     int n_sats, int K_max, const int32_t *K_sat, int adaptive, int n_sub, double rtol,
                                     double atol, double max_step, double *out_host, int32_t *status_host,
                                     int32_t *n_nodes_host)
{
    if (!K_sat) return fail(MPC_E_INVALID, "null K_sat");
    const AdaptiveOpts o{rtol, atol, max_step, nullptr};
    return disc_host(ctx, x, u, tf, p, n_sats, K_max, adaptive ? 1 : n_sub, adaptive ? &o : nullptr, out_host, status_host,
                     adaptive ? n_nodes_host : nullptr, K_sat);
}

int mpc_discretize_batch_adaptive_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf,
                                       const mpc_params *p, int n_sats, int K, double rtol, double atol,
                                       double max_step, double *out_host, int32_t *status_host, int32_t *n_nodes_host)
{
    const AdaptiveOpts o{rtol, atol, max_step, nullptr};
    return disc_host(ctx, x, u, tf, p, n_sats, K, 1, &o, out_host, status_host, n_nodes_host);
}

int mpc_discretize_batch_ugrid_host(mpc_ctx *ctx, const double *x, const double *u, int u_cols, const double *tf,
                                    const mpc_params *p, int n_sats, int K, int adaptive, int n_sub, double rtol,
                                    double atol, double max_step, double *out_host, int32_t *status_host,
                                    int32_t *n_nodes_host)
{
    if (u_cols < 2) return fail(MPC_E_INVALID, "u needs at least 2 columns (got %d)", u_cols);
    UcolsScope scope(u_cols);
    const AdaptiveOpts o{rtol, atol, max_step, nullptr};
    return disc_host(ctx, x, u, tf, p, n_sats, K, adaptive ? 1 : n_sub, adaptive ? &o : nullptr, out_host, status_host,
                     adaptive ? n_nodes_host : nullptr);
}

static int upload_table(mpc_ctx *ctx, const mpc_controller *ctrl, int n_sats, cudaStream_t st)
{
    if (ctrl->kind != MPC_CTRL_SEQUENCE) return MPC_SUCCESS;
    const size_t cnt = (size_t)(ctrl->table_per_sat ? n_sats : 1) * 3 * ctrl->table_len;
    int rc = ensure(ctx->d_tab, ctx->cap_tab, cnt);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_tab, ctrl->table, cnt * sizeof(double), cudaMemcpyHostToDevice, st));
    if (ctrl->end_tau_per_sat) {
        if ((rc = ensure(ctx->d_endtau, ctx->cap_endtau, (size_t)n_sats))) return rc;
        CUDA_TRY(cudaMemcpyAsync(ctx->d_endtau, ctrl->end_tau_per_sat, (size_t)n_sats * sizeof(double),
                                 cudaMemcpyHostToDevice, st));
    }
    return MPC_SUCCESS;
}

// T_sat != nullptr: per-satellite sample counts (T = Tmax) and table lengths (ku, may be NULL), host arrays
// (mpc_propagate_batch_rk45_ragged_host)
// consts != nullptr: per-satellite constants (mpc_propagate_batch_rk45_units_host)
static int prop_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p, const mpc_controller *ctrl,
                     int n_sats, int T, PropMode mode, double *y_host, double *u_host, int32_t *status_host,
                     int32_t *n_steps_host, const int32_t *T_sat = nullptr, const int32_t *ku_in = nullptr,
                     const mpc_sat_consts *consts = nullptr, const mpc_atmosphere *atmo = nullptr)
{
    if (!ctx || !y0 || !tf || !p || !y_host) return fail(MPC_E_INVALID, "null pointer argument");
    if (n_sats < 0 || T < 0 || mode.n_sub < 0) return fail(MPC_E_INVALID, "need n_sats >= 0, T >= 0, n_sub >= 0");
    int rc = check_ctrl(ctrl);
    if (rc) return rc;
    const int32_t *ku = (ctrl->kind == MPC_CTRL_SEQUENCE) ? ku_in : nullptr;
    if (T_sat && (rc = check_counts(T_sat, n_sats, T, "T_sat"))) return rc;
    if (ku && (rc = check_counts(ku, n_sats, ctrl->table_len, "table_len_sat"))) return rc;
    if (consts && (rc = check_sat_consts(consts, n_sats))) return rc;
    if (atmo && (rc = check_atmo(atmo, p, consts, n_sats))) return rc;
    if (n_sats == 0 || T == 0) return MPC_SUCCESS;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if ((rc = ensure(ctx->d_y0, ctx->cap_y0, (size_t)n_sats * 7))) return rc;
    if ((rc = ensure(ctx->d_tf, ctx->cap_tf, (size_t)n_sats))) return rc;
    if ((rc = ensure(ctx->d_x, ctx->cap_x, (size_t)n_sats * 7 * T))) return rc;
    if ((rc = ensure(ctx->d_u, ctx->cap_u, (size_t)n_sats * 3 * T))) return rc;
    if ((rc = ensure(ctx->d_status2, ctx->cap_status2, (size_t)n_sats))) return rc;
    cudaStream_t st = ctx->s_compute;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_y0, y0, (size_t)n_sats * 7 * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_tf, tf, (size_t)n_sats * sizeof(double), cudaMemcpyHostToDevice, st));
    if ((rc = upload_table(ctx, ctrl, n_sats, st))) return rc;
    if (mode.rk45() && n_steps_host) {
        if ((rc = ensure(ctx->d_nodes, ctx->cap_nodes, (size_t)n_sats))) return rc;
        mode.n_steps = ctx->d_nodes;
    }
    if (T_sat || ku) {
        if ((rc = ensure(ctx->d_cnt, ctx->cap_cnt, (size_t)n_sats * 2))) return rc;
        if (T_sat) CUDA_TRY(cudaMemcpyAsync(ctx->d_cnt, T_sat, (size_t)n_sats * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        if (ku) CUDA_TRY(cudaMemcpyAsync(ctx->d_cnt + n_sats, ku, (size_t)n_sats * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    }
    if (T_sat) {   // the kernel leaves the padding columns alone: they go back as NaN (all-ones bytes)
        CUDA_TRY(cudaMemsetAsync(ctx->d_x, 0xFF, (size_t)n_sats * 7 * T * sizeof(double), st));
        if (u_host) CUDA_TRY(cudaMemsetAsync(ctx->d_u, 0xFF, (size_t)n_sats * 3 * T * sizeof(double), st));
    }
    if (consts) {
        if ((rc = ensure(ctx->d_psc, ctx->cap_psc, (size_t)n_sats * MPC_SAT_SCRATCH_DOUBLES))) return rc;
        if (atmo) {
            const double r_earth = atmo->r_earth;
            rc = upload_sat_table<mpc::AtmoSat>(p, consts, n_sats, ctx->d_psc, st,
                                                [r_earth](const mpc_params *q) { return atmo_sat(q, r_earth); });
        } else {
            rc = upload_sat_table<mpc::PropParams>(p, consts, n_sats, ctx->d_psc, st, prop_params);
        }
        if (rc) return rc;
    }
    const mpc::AtmoParams A = atmo ? atmo_params(atmo, atmo->r_earth / p->r_e) : mpc::AtmoParams{};
    if ((rc = prop_device(ctx->d_y0, ctx->d_tf, p, ctrl, ctx->d_tab, ctrl->end_tau_per_sat ? ctx->d_endtau : nullptr, n_sats, T, mode,
                          ctx->d_x, ctx->d_u, ctx->d_status2, st, nullptr, 0, nullptr, T_sat ? ctx->d_cnt : nullptr,
                          ku ? ctx->d_cnt + n_sats : nullptr, consts ? ctx->d_psc : nullptr, atmo ? &A : nullptr)))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(y_host, ctx->d_x, (size_t)n_sats * 7 * T * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (u_host) CUDA_TRY(cudaMemcpyAsync(u_host, ctx->d_u, (size_t)n_sats * 3 * T * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (status_host)
        CUDA_TRY(cudaMemcpyAsync(status_host, ctx->d_status2, (size_t)n_sats * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (mode.rk45() && n_steps_host)
        CUDA_TRY(cudaMemcpyAsync(n_steps_host, ctx->d_nodes, (size_t)n_sats * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return MPC_SUCCESS;
}

int mpc_propagate_batch_rk45_ragged_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                                         const mpc_controller *ctrl, int n_sats, int T_max, const int32_t *T_sat,
                                         const int32_t *table_len_sat, double rtol, double atol, double max_step,
                                         double *y_host, double *u_host, int32_t *status_host, int32_t *n_steps_host)
{
    if (!T_sat) return fail(MPC_E_INVALID, "null T_sat");
    PropMode m;
    m.rk = mpc::Rk45Opts{rtol, atol, max_step};
    return prop_host(ctx, y0, tf, p, ctrl, n_sats, T_max, m, y_host, u_host, status_host, n_steps_host, T_sat, table_len_sat);
}

// ---- per-satellite designer units --------------------------------------------------------------------------------------
int mpc_discretize_batch_units(const double *x, const double *u, const double *tf, const mpc_params *p,
                               const mpc_sat_consts *consts, int n_sats, int K_max, const int32_t *K_sat, int64_t *first,
                               double *consts_scratch, int adaptive, int n_sub, double rtol, double atol, double max_step,
                               double *out, int64_t out_pitch, int64_t out_offset, int32_t *status, int32_t *n_nodes,
                               void *stream)
{
    int rc = check_units_disc(x, u, tf, p, consts, n_sats, K_max, K_sat, adaptive, n_sub, rtol, atol, max_step);
    if (rc) return rc;
    if (!out || (K_sat && !first)) return fail(MPC_E_INVALID, "null output / first");
    if (out_pitch < out_offset + (long long)n_sats * (K_max - 1) || out_offset < 0)
        return fail(MPC_E_INVALID, "out_pitch/out_offset do not hold the batch");
    if (n_sats == 0) return MPC_SUCCESS;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = upload_sat_table<mpc::DiscParams>(p, consts, n_sats, consts_scratch, st, disc_params))) return rc;
    long long n_units = (long long)n_sats * (K_max - 1);
    // the fixed-step form of a rectangular batch is the ragged launch with equal counts (launch_units_disc); its prefix
    // sums go behind the table in the scratch (3 + 1 of the MPC_SAT_SCRATCH_DOUBLES per satellite, plus one)
    std::vector<int32_t> equal;
    if (!K_sat && !adaptive) {
        equal.assign((size_t)n_sats, K_max);
        K_sat = equal.data();
        first = (int64_t *)(consts_scratch + (size_t)n_sats * (sizeof(mpc::DiscParams) / sizeof(double)));
    }
    if (K_sat) {
        const std::vector<long long> f = ragged_first(K_sat, n_sats);
        CUDA_TRY(cudaMemcpyAsync(first, f.data(), f.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
        n_units = f[n_sats];
    }
    mpc::DstTab tab{};
    tab.p[0] = out;
    const AdaptiveOpts o{rtol, atol, max_step, n_nodes};
    return launch_units_disc(x, u, tf, (const mpc::DiscParams *)consts_scratch, p->include_j2, n_sats, K_max, n_units,
                             K_sat ? (const long long *)first : nullptr, adaptive ? &o : nullptr, n_sub, tab, out_pitch,
                             out_offset, status, st);
}

// ---- one rank's shard of a ragged batch, stored into every rank's gathered buffer ----------------------------------------
int mpc_discretize_batch_ragged_gather(const double *x, const double *u, const double *tf, const mpc_params *p,
                                       const mpc_sat_consts *consts, int n_sats, int K_cap, const int32_t *K_sat, int64_t *first,
                                       double *consts_scratch, int adaptive, int n_sub, double rtol, double atol,
                                       double max_step, double *const *dst, int n_dst, int64_t out_pitch, int64_t out_offset,
                                       int skip_const, int32_t *status, int32_t *n_nodes, void *stream)
{
    int rc = consts ? check_units_disc(x, u, tf, p, consts, n_sats, K_cap, K_sat, adaptive, n_sub, rtol, atol, max_step)
                    : check_ragged_disc(x, u, tf, p, n_sats, K_cap, K_sat, adaptive, n_sub, rtol, atol, max_step);
    if (rc) return rc;
    if (!K_sat || !first) return fail(MPC_E_INVALID, "null K_sat / first");
    if (!dst || (n_dst != 1 && n_dst != 2 && n_dst != 4 && n_dst != 8))
        return fail(MPC_E_INVALID, "n_dst must be 1, 2, 4 or 8 (got %d)", n_dst);
    for (int d = 0; d < n_dst; ++d)
        if (!dst[d]) return fail(MPC_E_INVALID, "null destination %d", d);
    if (skip_const < 0 || skip_const > 2) return fail(MPC_E_INVALID, "skip_const must be 0, 1 or 2 (got %d)", skip_const);
    if (out_pitch < out_offset + (long long)n_sats * (K_cap - 1) || out_offset < 0)
        return fail(MPC_E_INVALID, "out_pitch/out_offset do not hold the batch");
    if (n_sats == 0) return MPC_SUCCESS;
    cudaStream_t st = (cudaStream_t)stream;
    if (consts && (rc = upload_sat_table<mpc::DiscParams>(p, consts, n_sats, consts_scratch, st, disc_params))) return rc;
    const std::vector<long long> f = ragged_first(K_sat, n_sats);
    CUDA_TRY(cudaMemcpyAsync(first, f.data(), f.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    const long long *fd = (const long long *)first;
    mpc::DstTab tab{};
    for (int d = 0; d < n_dst; ++d) tab.p[d] = dst[d];
    tab.skip_const = skip_const;
    const AdaptiveOpts o{rtol, atol, max_step, n_nodes};
    const AdaptiveOpts *ad = adaptive ? &o : nullptr;
    const mpc::DiscParams P = disc_params(p);
    if (n_dst == 1) {   // the single-GPU launches
        if (consts)
            return launch_units_disc(x, u, tf, (const mpc::DiscParams *)consts_scratch, p->include_j2, n_sats, K_cap, f[n_sats], fd,
                                     ad, n_sub, tab, out_pitch, out_offset, status, st);
        return p->include_j2 ? launch_ragged<true>(x, u, tf, P, n_sats, K_cap, f[n_sats], fd, ad, n_sub, tab, out_pitch, out_offset, status, st)
                             : launch_ragged<false>(x, u, tf, P, n_sats, K_cap, f[n_sats], fd, ad, n_sub, tab, out_pitch, out_offset, status, st);
    }
    // the block sizes launch_ragged / launch_units_disc choose from the live count (default mode: 32 or 256 threads, the
    // 128-thread CTA of mpc_set_tuning(21) has no multi-destination build)
    tab.em = em_level();
    MpcUnitsDisc a{};
    a.x = x;
    a.u = u;
    a.tf = tf;
    a.psc = consts ? consts_scratch : nullptr;
    a.dst_tab = &tab;
    a.first = fd;
    a.n_units = f[n_sats];
    a.include_j2 = p->include_j2;
    a.n_sats = n_sats;
    a.K = K_cap;
    a.n_sub = n_sub;
    a.adaptive = adaptive;
    if (adaptive) {
        a.block = a.n_units < 148LL * 256 ? 32 : 256;
        a.rtol = rtol;
        a.atol = atol;
        a.max_step = max_step;
        a.n_nodes = n_nodes;
    } else {
        a.block = (a.n_units > 148LL * 32 && a.n_units <= 148LL * 128) || a.n_units >= 148LL * 9 * 32 * 2 ? kDiscBlock : 32;
    }
    a.pitch = out_pitch;
    a.offset = out_offset;
    a.status = status;
    a.stream = st;
    CUDA_TRY(mpc_shard_launch_disc(&a, &P, n_dst));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return MPC_SUCCESS;
}

int mpc_discretize_batch_units_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf, const mpc_params *p,
                                    const mpc_sat_consts *consts, int n_sats, int K_max, const int32_t *K_sat, int adaptive,
                                    int n_sub, double rtol, double atol, double max_step, double *out_host,
                                    int32_t *status_host, int32_t *n_nodes_host)
{
    if (!consts) return fail(MPC_E_INVALID, "null consts");
    const AdaptiveOpts o{rtol, atol, max_step, nullptr};
    std::vector<int32_t> equal;   // a rectangular fixed-step batch: the ragged launch with equal counts (launch_units_disc)
    if (!K_sat && !adaptive && n_sats > 0) {
        equal.assign((size_t)n_sats, K_max);
        K_sat = equal.data();
    }
    return disc_host(ctx, x, u, tf, p, n_sats, K_max, adaptive ? 1 : n_sub, adaptive ? &o : nullptr, out_host, status_host,
                     adaptive ? n_nodes_host : nullptr, K_sat, consts);
}

// ---- the default quadrature mode with scipy's RK23 ---------------------------------------------------------------------
int mpc_discretize_batch_rk23(const double *x, const double *u, const double *tf, const mpc_params *p,
                              const mpc_sat_consts *consts, int n_sats, int K_max, const int32_t *K_sat, int64_t *first,
                              double *consts_scratch, double rtol, double atol, double max_step, double *out, int64_t out_pitch,
                              int64_t out_offset, int32_t *status, int32_t *n_nodes, void *stream)
{
    int rc = check_rk23_disc(x, u, tf, p, consts, n_sats, K_max, K_sat, rtol, atol, max_step);
    if (rc) return rc;
    if (!out || (K_sat && !first)) return fail(MPC_E_INVALID, "null output / first");
    if (out_pitch < out_offset + (long long)n_sats * (K_max - 1) || out_offset < 0)
        return fail(MPC_E_INVALID, "out_pitch/out_offset do not hold the batch");
    if (n_sats == 0) return MPC_SUCCESS;
    cudaStream_t st = (cudaStream_t)stream;
    if (consts && (rc = upload_sat_table<mpc::DiscParams>(p, consts, n_sats, consts_scratch, st, disc_params))) return rc;
    long long n_units = (long long)n_sats * (K_max - 1);
    if (K_sat) {
        const std::vector<long long> f = ragged_first(K_sat, n_sats);
        CUDA_TRY(cudaMemcpyAsync(first, f.data(), f.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
        n_units = f[n_sats];
    }
    const AdaptiveOpts o{rtol, atol, max_step, n_nodes};
    return launch_rk23(x, u, tf, disc_params(p), consts ? (const mpc::DiscParams *)consts_scratch : nullptr, p->include_j2,
                       n_sats, K_max, n_units, K_sat ? (const long long *)first : nullptr, o, out, out_pitch, out_offset,
                       status, st);
}

int mpc_discretize_batch_rk23_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf, const mpc_params *p,
                                   const mpc_sat_consts *consts, int n_sats, int K_max, const int32_t *K_sat, double rtol,
                                   double atol, double max_step, double *out_host, int32_t *status_host,
                                   int32_t *n_nodes_host)
{
    AdaptiveOpts o{rtol, atol, max_step, nullptr};
    o.rk23 = 1;
    return disc_host(ctx, x, u, tf, p, n_sats, K_max, 1, &o, out_host, status_host, n_nodes_host, K_sat, consts);
}

// ---- conjunction screening (mpc_screen_conjunctions[_host]; mpc_b200_conj.cu) -------------------------------------------

static int check_conj(const double *y, int n_sats, int T, const double *scale, double duration, double threshold)
{
    if (!y || !scale) return fail(MPC_E_INVALID, "null y / scale");
    if (n_sats < 2 || T < 2) return fail(MPC_E_INVALID, "need n_sats >= 2 and T >= 2 (got %d, %d)", n_sats, T);
    if (!(std::isfinite(duration) && duration > 0.0)) return fail(MPC_E_INVALID, "need a finite duration > 0 (got %g)", duration);
    if (!(std::isfinite(threshold) && threshold > 0.0))
        return fail(MPC_E_INVALID, "need a finite threshold > 0 (got %g)", threshold);
    for (int s = 0; s < n_sats; ++s)
        for (int c = 0; c < 2; ++c)
            if (!(std::isfinite(scale[2 * s + c]) && scale[2 * s + c] > 0.0))
                return fail(MPC_E_INVALID, "scale[%d][%d] = %g: every scale must be finite and > 0", s, c, scale[2 * s + c]);
    if (mpc_conj_record_size() != sizeof(mpc_conjunction))
        return fail(MPC_E_CUDA, "mpc_b200_conj.cu was built against a different event record");
    return MPC_SUCCESS;
}

int64_t mpc_conjunction_scratch_doubles(int n_sats, int T)
{
    return n_sats < 0 || T < 2 ? 0 : (int64_t)mpc_conj_scratch_doubles(n_sats, T);
}

int mpc_screen_conjunctions(const double *y, int n_sats, int T, const double *scale, double duration, double threshold,
                            double *scratch, mpc_conjunction *events, int64_t capacity, uint64_t *counters,
                            int32_t *skipped, void *stream)
{
    int rc = check_conj(y, n_sats, T, scale, duration, threshold);
    if (rc) return rc;
    if (!scratch || !counters || !skipped || capacity < 0 || (capacity > 0 && !events))
        return fail(MPC_E_INVALID, "null scratch / counters / skipped, or no events buffer for capacity %lld", (long long)capacity);
    MpcConjLaunch a{y, scratch, scale, n_sats, T, duration / (T - 1), threshold, events, capacity,
                    (unsigned long long *)counters, skipped, (cudaStream_t)stream};
    CUDA_TRY(mpc_conj_launch(&a));
    g_launches.fetch_add(2, std::memory_order_relaxed);
    return MPC_SUCCESS;
}

int mpc_screen_conjunctions_host(mpc_ctx *ctx, const double *y, int n_sats, int T, const double *scale, double duration,
                                 double threshold, mpc_conjunction *events_host, int64_t capacity, int64_t *count,
                                 int64_t *n_flagged, int32_t *skipped_host)
{
    if (!ctx || !count || !n_flagged || !skipped_host || capacity < 0 || (capacity > 0 && !events_host))
        return fail(MPC_E_INVALID, "null ctx / count / n_flagged / skipped, or no events buffer for capacity %lld", (long long)capacity);
    int rc = check_conj(y, n_sats, T, scale, duration, threshold);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const size_t ev_doubles = (size_t)std::max<int64_t>(capacity, 1) * (sizeof(mpc_conjunction) / sizeof(double));
    if ((rc = ensure(ctx->d_x, ctx->cap_x, (size_t)n_sats * 7 * T))) return rc;
    if ((rc = ensure(ctx->d_conj, ctx->cap_conj, (size_t)mpc_conj_scratch_doubles(n_sats, T)))) return rc;
    if ((rc = ensure(ctx->d_conj_ev, ctx->cap_conj_ev, ev_doubles))) return rc;
    if ((rc = ensure(ctx->d_conj_cnt, ctx->cap_conj_cnt, 2))) return rc;
    if ((rc = ensure(ctx->d_status, ctx->cap_status, (size_t)n_sats))) return rc;
    cudaStream_t st = ctx->s_compute;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_x, y, (size_t)n_sats * 7 * T * sizeof(double), cudaMemcpyHostToDevice, st));
    MpcConjLaunch a{ctx->d_x, ctx->d_conj, scale, n_sats, T, duration / (T - 1), threshold, ctx->d_conj_ev, capacity,
                    ctx->d_conj_cnt, ctx->d_status, st};
    CUDA_TRY(mpc_conj_launch(&a));
    g_launches.fetch_add(2, std::memory_order_relaxed);
    unsigned long long cnt[2];
    CUDA_TRY(cudaMemcpyAsync(cnt, ctx->d_conj_cnt, sizeof cnt, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(skipped_host, ctx->d_status, (size_t)n_sats * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const long long n_out = std::min<long long>((long long)cnt[0], capacity);
    if (n_out > 0) {
        CUDA_TRY(cudaMemcpyAsync(events_host, ctx->d_conj_ev, (size_t)n_out * sizeof(mpc_conjunction), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    *count = (int64_t)cnt[0];
    *n_flagged = (int64_t)cnt[1];
    return MPC_SUCCESS;
}

int mpc_propagate_batch_rk45_units(const double *y0, const double *tf, const mpc_params *p, const mpc_sat_consts *consts,
                                   const mpc_controller *ctrl, int n_sats, int T_max, const int32_t *T_sat,
                                   const int32_t *table_len_sat, double *consts_scratch, double rtol, double atol,
                                   double max_step, double *y, double *u_out, int32_t *status, int32_t *n_steps,
                                   void *stream)
{
    if (!p) return fail(MPC_E_INVALID, "null pointer argument");
    if (T_sat && T_max < 2) return fail(MPC_E_INVALID, "need T_max >= 2 (got %d)", T_max);
    int rc = check_sat_consts(consts, n_sats);
    if (rc) return rc;
    if (n_sats > 0 && T_max > 0 &&
        (rc = upload_sat_table<mpc::PropParams>(p, consts, n_sats, consts_scratch, (cudaStream_t)stream, prop_params)))
        return rc;
    PropMode m;
    m.rk = mpc::Rk45Opts{rtol, atol, max_step};
    m.n_steps = n_steps;
    return prop_device(y0, tf, p, ctrl, ctrl ? ctrl->table : nullptr, ctrl ? ctrl->end_tau_per_sat : nullptr, n_sats, T_max, m,
                       y, u_out, status, (cudaStream_t)stream, nullptr, 0, nullptr, T_sat, table_len_sat,
                       (const mpc::PropParams *)consts_scratch);
}

int mpc_propagate_batch_rk45_units_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                                        const mpc_sat_consts *consts, const mpc_controller *ctrl, int n_sats, int T_max,
                                        const int32_t *T_sat, const int32_t *table_len_sat, double rtol, double atol,
                                        double max_step, double *y_host, double *u_host, int32_t *status_host,
                                        int32_t *n_steps_host)
{
    if (!consts) return fail(MPC_E_INVALID, "null consts");
    PropMode m;
    m.rk = mpc::Rk45Opts{rtol, atol, max_step};
    return prop_host(ctx, y0, tf, p, ctrl, n_sats, T_max, m, y_host, u_host, status_host, n_steps_host, T_sat, table_len_sat,
                     consts);
}

int mpc_propagate_batch_rk45_atmo(const double *y0, const double *tf, const mpc_params *p, const mpc_sat_consts *consts,
                                  const mpc_controller *ctrl, int n_sats, int T_max, const int32_t *T_sat,
                                  const int32_t *table_len_sat, double *consts_scratch, double rtol, double atol,
                                  double max_step, double *y, double *u_out, int32_t *status, int32_t *n_steps,
                                  const mpc_atmosphere *atmo, void *stream)
{
    if (!p) return fail(MPC_E_INVALID, "null pointer argument");
    if (T_sat && T_max < 2) return fail(MPC_E_INVALID, "need T_max >= 2 (got %d)", T_max);
    int rc = consts ? check_sat_consts(consts, n_sats) : MPC_SUCCESS;
    if (rc || (rc = check_atmo(atmo, p, consts, n_sats))) return rc;
    if (consts && n_sats > 0 && T_max > 0) {
        const double r_earth = atmo->r_earth;
        if ((rc = upload_sat_table<mpc::AtmoSat>(p, consts, n_sats, consts_scratch, (cudaStream_t)stream,
                                                 [r_earth](const mpc_params *q) { return atmo_sat(q, r_earth); })))
            return rc;
    }
    const mpc::AtmoParams A = atmo_params(atmo, atmo->r_earth / p->r_e);
    PropMode m;
    m.rk = mpc::Rk45Opts{rtol, atol, max_step};
    m.n_steps = n_steps;
    return prop_device(y0, tf, p, ctrl, ctrl ? ctrl->table : nullptr, ctrl ? ctrl->end_tau_per_sat : nullptr, n_sats, T_max, m,
                       y, u_out, status, (cudaStream_t)stream, nullptr, 0, nullptr, T_sat, table_len_sat,
                       consts ? consts_scratch : nullptr, &A);
}

int mpc_propagate_batch_rk45_atmo_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                                       const mpc_sat_consts *consts, const mpc_controller *ctrl, int n_sats, int T_max,
                                       const int32_t *T_sat, const int32_t *table_len_sat, double rtol, double atol,
                                       double max_step, double *y_host, double *u_host, int32_t *status_host,
                                       int32_t *n_steps_host, const mpc_atmosphere *atmo)
{
    if (!atmo) return fail(MPC_E_INVALID, "null atmosphere");
    PropMode m;
    m.rk = mpc::Rk45Opts{rtol, atol, max_step};
    return prop_host(ctx, y0, tf, p, ctrl, n_sats, T_max, m, y_host, u_host, status_host, n_steps_host, T_sat, table_len_sat,
                     consts, atmo);
}

int mpc_propagate_batch_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                             const mpc_controller *ctrl, int n_sats, int T, int n_sub, double *y_host,
                             double *u_host, int32_t *status_host)
{
    return prop_host(ctx, y0, tf, p, ctrl, n_sats, T, mode_of(n_sub), y_host, u_host, status_host, nullptr);
}

int mpc_propagate_batch_rk45_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                                  const mpc_controller *ctrl, int n_sats, int T, double rtol, double atol,
                                  double max_step, double *y_host, double *u_host, int32_t *status_host,
                                  int32_t *n_steps_host)
{
    PropMode m;
    m.rk = mpc::Rk45Opts{rtol, atol, max_step};
    return prop_host(ctx, y0, tf, p, ctrl, n_sats, T, m, y_host, u_host, status_host, n_steps_host);
}

int mpc_propagate_discretize_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                                  const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T,
                                  int n_sub_prop, int n_sub_disc, double *y_host, double *u_host,
                                  double *out_host, int32_t *status_host)
{
    if (!ctx || !y0 || !tf || !p_prop || !p_disc || !out_host) return fail(MPC_E_INVALID, "null pointer argument");
    const int K = T;
    if (n_sats < 0 || K < 2 || n_sub_prop < 0 || n_sub_disc < 1) return fail(MPC_E_INVALID, "need n_sats >= 0, T >= 2, n_sub_prop >= 0, n_sub_disc >= 1");
    if (p_disc->include_drag && !(p_disc->disc_cd > 0.0 && p_disc->disc_rho >= 0.0))
        return fail(MPC_E_UNSUPPORTED, "include_drag needs disc_cd / disc_rho (const.CD, rho_func): the reference raises without them too");
    if (int rcm = check_drag_model(p_disc)) return rcm;
    int rc = check_ctrl(ctrl);
    if (rc) return rc;
    if (n_sats == 0) return MPC_SUCCESS;
    const long long n_int = (long long)n_sats * (K - 1);
    CUDA_TRY(cudaSetDevice(ctx->device));
    if ((rc = ensure(ctx->d_y0, ctx->cap_y0, (size_t)n_sats * 7))) return rc;
    if ((rc = ensure(ctx->d_tf, ctx->cap_tf, (size_t)n_sats))) return rc;
    if ((rc = ensure(ctx->d_x, ctx->cap_x, (size_t)n_sats * 7 * K))) return rc;
    if ((rc = ensure(ctx->d_u, ctx->cap_u, (size_t)n_sats * 3 * K))) return rc;
    if ((rc = ensure(ctx->d_out, ctx->cap_out, (size_t)n_int * MPC_OUT_ROWS))) return rc;
    if ((rc = ensure(ctx->d_status, ctx->cap_status, (size_t)n_int))) return rc;
    if ((rc = ensure(ctx->d_status2, ctx->cap_status2, (size_t)n_sats))) return rc;
    const int cs = chunk_sats(ctx, n_sats, K);
    const int n_chunks = (n_sats + cs - 1) / cs;
    if ((rc = ensure_events(ctx, (size_t)n_chunks))) return rc;
    cudaStream_t st = ctx->s_compute;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_y0, y0, (size_t)n_sats * 7 * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_tf, tf, (size_t)n_sats * sizeof(double), cudaMemcpyHostToDevice, st));
    if ((rc = upload_table(ctx, ctrl, n_sats, st))) return rc;
    // the whole batch is propagated first (one thread per satellite is latency-bound: chunking it
    // would only serialise the latency), then discretized chunk by chunk while results stream out
    if ((rc = prop_device(ctx->d_y0, ctx->d_tf, p_prop, ctrl, ctx->d_tab, ctrl->end_tau_per_sat ? ctx->d_endtau : nullptr, n_sats, K,
                          mode_of(n_sub_prop), ctx->d_x, ctx->d_u,
                          ctx->d_status2, st)))
        return rc;
    // the reference trajectory and inputs go back to the host while the first chunks are being discretized
    if ((rc = ensure_events(ctx, (size_t)n_chunks + 1))) return rc;
    CUDA_TRY(cudaEventRecord(ctx->ev[n_chunks], st));
    CUDA_TRY(cudaStreamWaitEvent(ctx->s_copy, ctx->ev[n_chunks], 0));
    if (y_host) CUDA_TRY(cudaMemcpyAsync(y_host, ctx->d_x, (size_t)n_sats * 7 * K * sizeof(double), cudaMemcpyDeviceToHost, ctx->s_copy));
    if (u_host) CUDA_TRY(cudaMemcpyAsync(u_host, ctx->d_u, (size_t)n_sats * 3 * K * sizeof(double), cudaMemcpyDeviceToHost, ctx->s_copy));
    const mpc::DiscParams P = disc_params(p_disc);
    for (int c = 0; c < n_chunks; ++c) {
        const int s0 = c * cs, ns = std::min(cs, n_sats - s0);
        mpc::DstTab tab{};
        tab.p[0] = ctx->d_out;
        const long long off = (long long)s0 * (K - 1);
        rc = launch_fixed(ctx->d_x + (size_t)s0 * 7 * K, ctx->d_u + (size_t)s0 * 3 * K, ctx->d_tf + s0, p_disc, P, ns, K,
                          n_sub_disc, tab, n_int, off, ctx->d_status + off, st);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(ctx->ev[c], st));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_copy, ctx->ev[c], 0));
        if ((rc = copy_out_chunk(out_host, ctx->d_out, n_int, off, (long long)ns * (K - 1), ctx->s_copy))) return rc;
    }
    fill_const_rows(out_host, n_int);   // host writes the structural constants while the GPU / DMA engine work
    if (status_host) {   // int32 words through pinned staging (see disc_host)
        if ((rc = ensure_stage(ctx, (size_t)n_int + n_sats))) return rc;
        CUDA_TRY(cudaMemcpyAsync(is_pinned(status_host) ? status_host : ctx->h_stage, ctx->d_status, (size_t)n_int * sizeof(int32_t),
                                 cudaMemcpyDeviceToHost, ctx->s_copy));
        CUDA_TRY(cudaMemcpyAsync(ctx->h_stage + n_int, ctx->d_status2, (size_t)n_sats * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->s_copy));
    }
    CUDA_TRY(cudaStreamSynchronize(ctx->s_copy));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (status_host) {
        if (!is_pinned(status_host)) memcpy(status_host, ctx->h_stage, (size_t)n_int * sizeof(int32_t));
        // a satellite whose propagation failed poisons its intervals: surface it in the interval status
        const int32_t *ps = ctx->h_stage + n_int;
        for (int s = 0; s < n_sats; ++s)
            if (ps[s])
                for (int k = 0; k < K - 1; ++k) status_host[(size_t)s * (K - 1) + k] = ps[s];
    }
    return MPC_SUCCESS;
}

}  // extern "C"

// ------------------------------------------------------------------------- overlapped propagate -> discretize
// One SCP linearization pass on device buffers (control.py:180-188: propagate -> extract_uk -> discretize) with the
// propagation HIDDEN behind the discretization.  The propagation is sequential in tau and latency-bound (a handful of
// warps, ~0.56 ms whatever the batch), the discretization fills the machine for milliseconds and interval k only needs
// the samples k and k+1.  So the intervals are cut into n_windows windows along k; the propagation kernel publishes a
// per-window progress word, and window b's discretization kernel is gated on it by a stream memory operation
// (cuStreamWaitValue32) -- the dependency is resolved by the stream front end, no CTA ever spins on a flag, nothing can
// deadlock.  Windows alternate over two streams so that the tail of one overlaps the head of the next.  Same kernels,
// same arithmetic: the result is bit-identical to mpc_propagate_batch followed by mpc_discretize_batch.
namespace {

constexpr int kMaxWindows = 64;

typedef CUresult (*StreamWaitValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);

StreamWaitValue32Fn stream_wait_value32()
{
    static StreamWaitValue32Fn fn = [] {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            f = nullptr;
        }
        return (StreamWaitValue32Fn)f;
    }();
    return fn;
}

int ensure_overlap(mpc_ctx *ctx)
{
    // every resource on its own, so that a failure half way leaves nothing to leak or to create twice
    for (cudaStream_t &w : ctx->s_win)
        if (!w) CUDA_TRY(cudaStreamCreateWithFlags(&w, cudaStreamNonBlocking));
    for (cudaEvent_t &e : ctx->ev_ov)
        if (!e) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    if (!ctx->d_progress) CUDA_TRY(cudaMalloc((void **)&ctx->d_progress, kMaxWindows * sizeof(unsigned int)));
    if (!ctx->s_prop) {
        int lo = 0, hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&ctx->s_prop, cudaStreamNonBlocking, hi));
    }
    return MPC_SUCCESS;
}

}  // namespace

namespace {

template <bool J2>
int launch_window(int n_dst, const double *x, const double *u, const double *tf, const mpc::DiscParams &P, int n_sats, int K,
                  int n_sub, const mpc::DstTab &tab, long long pitch, long long offset, int32_t *status, cudaStream_t st,
                  int k0, int kc)
{
    switch (n_dst) {
        case 1: return launch_pair_cfg<J2, kDiscBlock, 255, 1>(x, u, tf, P, n_sats, K, n_sub, tab, pitch, offset, status, st, k0, kc);
        case 2: return launch_pair_cfg<J2, kDiscBlock, 255, 2>(x, u, tf, P, n_sats, K, n_sub, tab, pitch, offset, status, st, k0, kc);
        case 4: return launch_pair_cfg<J2, kDiscBlock, 255, 4>(x, u, tf, P, n_sats, K, n_sub, tab, pitch, offset, status, st, k0, kc);
        case 8: return launch_pair_cfg<J2, kDiscBlock, 255, 8>(x, u, tf, P, n_sats, K, n_sub, tab, pitch, offset, status, st, k0, kc);
        default: return fail(MPC_E_INVALID, "n_dst must be 1, 2, 4 or 8 (got %d)", n_dst);
    }
}

int prop_disc_overlapped(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                         const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T, int n_sub_prop,
                         int n_sub_disc, double *x, double *u, double *const *dst, int n_dst, int64_t out_pitch,
                         int64_t out_offset, int32_t *status_prop, int32_t *status_disc, int n_windows, cudaStream_t st)
{
    if (!ctx || !y0 || !tf || !p_prop || !p_disc || !x || !u || !dst)
        return fail(MPC_E_INVALID, "null pointer argument");
    const int K = T;
    int rc = check_disc_args(x, u, tf, p_disc, n_sats, K, n_sub_disc);
    if (rc) return rc;
    if (n_sub_prop < 0) return fail(MPC_E_INVALID, "need n_sub_prop >= 0");
    if ((rc = check_ctrl(ctrl))) return rc;
    if (n_dst != 1 && n_dst != 2 && n_dst != 4 && n_dst != 8) return fail(MPC_E_INVALID, "n_dst must be 1, 2, 4 or 8 (got %d)", n_dst);
    for (int d = 0; d < n_dst; ++d)
        if (!dst[d]) return fail(MPC_E_INVALID, "null destination %d", d);
    const long long n_int = (long long)n_sats * (K - 1);
    if (out_pitch < out_offset + n_int || out_offset < 0) return fail(MPC_E_INVALID, "out_pitch/out_offset do not hold the batch");
    if (n_windows < 0 || n_windows > kMaxWindows) return fail(MPC_E_INVALID, "n_windows must be in [0, %d]", kMaxWindows);
    if (n_sats == 0) return MPC_SUCCESS;
    CUDA_TRY(cudaSetDevice(ctx->device));
    // Windows only pay when each of them still fills the machine (one wave = 2 CTAs of 128 threads per SM) and when the
    // two-node-step kernel runs (the windowed launch exists for it); otherwise the two kernels run back to back.
    const long long wave = (long long)ctx->sm_count * 2 * kDiscBlock;
    int nw = n_windows ? n_windows : 16;
    nw = (int)std::min<long long>(nw, std::min<long long>(n_int / wave, K - 1));
    const bool windowed = nw >= 2 && !p_disc->include_drag && g_pair.load(std::memory_order_relaxed) &&
                          g_tuning.load(std::memory_order_relaxed) == 0 && stream_wait_value32() != nullptr;
    const double *tab_dev = ctrl->table, *et_dev = ctrl->end_tau_per_sat;
    if (!windowed) {
        if ((rc = prop_device(y0, tf, p_prop, ctrl, tab_dev, et_dev, n_sats, K, mode_of(n_sub_prop), x, u, status_prop, st))) return rc;
        return disc_device(x, u, tf, p_disc, n_sats, K, n_sub_disc, dst, n_dst, out_pitch, out_offset, status_disc, st);
    }
    if ((rc = ensure_overlap(ctx))) return rc;
    const int seg = (K - 1 + nw - 1) / nw;         // intervals per window
    nw = (K - 1 + seg - 1) / seg;
    unsigned int gate = 0;   // value of progress[b] that opens window b
    CUDA_TRY(cudaMemsetAsync(ctx->d_progress, 0, kMaxWindows * sizeof(unsigned int), st));
    CUDA_TRY(cudaEventRecord(ctx->ev_ov[0], st));
    CUDA_TRY(cudaStreamWaitEvent(ctx->s_prop, ctx->ev_ov[0], 0));
    for (cudaStream_t w : ctx->s_win) CUDA_TRY(cudaStreamWaitEvent(w, ctx->ev_ov[0], 0));
    if ((rc = prop_device(y0, tf, p_prop, ctrl, tab_dev, et_dev, n_sats, K, mode_of(n_sub_prop), x, u, status_prop, ctx->s_prop,
                          ctx->d_progress, seg, &gate)))
        return rc;
    CUDA_TRY(cudaEventRecord(ctx->ev_ov[1], ctx->s_prop));   // propagation done: join of the caller's stream (and the gate of last resort)
    const mpc::DiscParams P = disc_params(p_disc);
    mpc::DstTab tab{};
    for (int d = 0; d < mpc::kMaxDst; ++d) tab.p[d] = (d < n_dst) ? dst[d] : nullptr;
    tab.skip_const = g_gather.active ? g_gather.skip_const : g_gather_skip_const.load(std::memory_order_relaxed);
    const int stagger = g_gather.active ? g_gather.stagger : g_gather_stagger.load(std::memory_order_relaxed);
    tab.km_ntot = g_gather.km_ntot;
    tab.km_soff = g_gather.km_soff;
    for (int b = 0; b < nw; ++b) {
        cudaStream_t sw = ctx->s_win[b & 1];
        const int k0 = b * seg, kc = std::min(seg, K - 1 - k0);
        // the staggered start of the fused all-gather (mpc_set_gather_tuning) belongs to the very first wave only
        tab.stagger_phases = (b == 0) ? stagger : 0;
        if (tab.stagger_phases > 1) {
            tab.first_wave_ctas = ctx->sm_count * 2;
            tab.stagger_cycles = (long long)n_sub_disc * 4940LL;
        }
        // gate: progress[b] == number of warps (RK4 propagator) / satellites (RK45 propagator).  Should the driver refuse the memory operation, the window waits for the
        // whole propagation instead (an ordinary event): coarser, still correct, nothing is left half enqueued.
        if (stream_wait_value32()((CUstream)sw, (CUdeviceptr)(uintptr_t)(ctx->d_progress + b), gate,
                                  CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS)
            CUDA_TRY(cudaStreamWaitEvent(sw, ctx->ev_ov[1], 0));
        rc = p_disc->include_j2
                 ? launch_window<true>(n_dst, x, u, tf, P, n_sats, K, n_sub_disc, tab, out_pitch, out_offset, status_disc, sw, k0, kc)
                 : launch_window<false>(n_dst, x, u, tf, P, n_sats, K, n_sub_disc, tab, out_pitch, out_offset, status_disc, sw, k0, kc);
        if (rc) return rc;
    }
    CUDA_TRY(cudaEventRecord(ctx->ev_ov[2], ctx->s_win[0]));
    CUDA_TRY(cudaEventRecord(ctx->ev_ov[3], ctx->s_win[1]));
    for (int e = 1; e < 4; ++e) CUDA_TRY(cudaStreamWaitEvent(st, ctx->ev_ov[e], 0));
    return MPC_SUCCESS;
}

}  // namespace

// Host-buffer pass in the k-major layout: windows along k gated on the propagation's progress, every finished window
// read back while the next one runs (see the header).
extern "C" int mpc_propagate_discretize_host_layout(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                                                    const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T,
                                                    int n_sub_prop, int n_sub_disc, double *y_host, double *u_host,
                                                    double *out_host, int32_t *status_host, int layout)
{
    if (layout == MPC_LAYOUT_SAT_MAJOR)
        return mpc_propagate_discretize_host(ctx, y0, tf, p_prop, p_disc, ctrl, n_sats, T, n_sub_prop, n_sub_disc, y_host, u_host,
                                             out_host, status_host);
    if (layout != MPC_LAYOUT_K_MAJOR) return fail(MPC_E_INVALID, "unknown layout %d", layout);
    if (!ctx || !y0 || !tf || !p_prop || !p_disc || !out_host) return fail(MPC_E_INVALID, "null pointer argument");
    const int K = T;
    if (n_sats < 0 || K < 2 || n_sub_prop < 0 || n_sub_disc < 1) return fail(MPC_E_INVALID, "need n_sats >= 0, T >= 2, n_sub_prop >= 0, n_sub_disc >= 1");
    if (p_disc->include_drag || !g_pair.load(std::memory_order_relaxed) || g_tuning.load(std::memory_order_relaxed) != 0)
        return fail(MPC_E_UNSUPPORTED, "the k-major layout is implemented by the two-node-step kernel only");
    int rc = check_ctrl(ctrl);
    if (rc) return rc;
    if (n_sats == 0) return MPC_SUCCESS;
    const long long n_int = (long long)n_sats * (K - 1);
    CUDA_TRY(cudaSetDevice(ctx->device));
    if ((rc = ensure(ctx->d_y0, ctx->cap_y0, (size_t)n_sats * 7))) return rc;
    if ((rc = ensure(ctx->d_tf, ctx->cap_tf, (size_t)n_sats))) return rc;
    if ((rc = ensure(ctx->d_x, ctx->cap_x, (size_t)n_sats * 7 * K))) return rc;
    if ((rc = ensure(ctx->d_u, ctx->cap_u, (size_t)n_sats * 3 * K))) return rc;
    if ((rc = ensure(ctx->d_out, ctx->cap_out, (size_t)n_int * MPC_OUT_ROWS))) return rc;
    if ((rc = ensure(ctx->d_status, ctx->cap_status, (size_t)n_int))) return rc;
    if ((rc = ensure(ctx->d_status2, ctx->cap_status2, (size_t)n_sats))) return rc;
    if ((rc = ensure_overlap(ctx))) return rc;
    // windows: each at least half a wave of the kernel (they alternate over two streams), at most g_host_windows (the
    // read-back of a window is what paces the pipeline; measured: profiles/r02_t_probe_e2e.txt)
    const long long wave = (long long)ctx->sm_count * 2 * kDiscBlock;
    int nw = (int)std::max<long long>(1, std::min<long long>(g_host_windows.load(std::memory_order_relaxed),
                                                           std::min<long long>(2 * n_int / wave, K - 1)));
    const bool gated = nw >= 2 && stream_wait_value32() != nullptr;
    if (!gated) nw = 1;
    const int seg = (K - 1 + nw - 1) / nw;
    nw = (K - 1 + seg - 1) / seg;
    if ((rc = ensure_events(ctx, (size_t)nw + 2))) return rc;
    cudaStream_t st = ctx->s_compute;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_y0, y0, (size_t)n_sats * 7 * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_tf, tf, (size_t)n_sats * sizeof(double), cudaMemcpyHostToDevice, st));
    if ((rc = upload_table(ctx, ctrl, n_sats, st))) return rc;
    CUDA_TRY(cudaMemsetAsync(ctx->d_progress, 0, kMaxWindows * sizeof(unsigned int), st));
    CUDA_TRY(cudaEventRecord(ctx->ev_ov[0], st));
    CUDA_TRY(cudaStreamWaitEvent(ctx->s_prop, ctx->ev_ov[0], 0));
    for (cudaStream_t w : ctx->s_win) CUDA_TRY(cudaStreamWaitEvent(w, ctx->ev_ov[0], 0));
    unsigned int gate = 0;
    const double *et_dev = ctrl->end_tau_per_sat ? ctx->d_endtau : nullptr;
    if ((rc = prop_device(ctx->d_y0, ctx->d_tf, p_prop, ctrl, ctx->d_tab, et_dev, n_sats, K, mode_of(n_sub_prop), ctx->d_x, ctx->d_u,
                          ctx->d_status2, ctx->s_prop, gated ? ctx->d_progress : nullptr, seg, &gate)))
        return rc;
    CUDA_TRY(cudaEventRecord(ctx->ev_ov[1], ctx->s_prop));
    const mpc::DiscParams P = disc_params(p_disc);
    mpc::DstTab tab{};
    tab.p[0] = ctx->d_out;
    tab.km_ntot = n_sats;
    tab.km_soff = 0;
    for (int b = 0; b < nw; ++b) {
        cudaStream_t sw = ctx->s_win[b & 1];
        const int k0 = b * seg, kc = std::min(seg, K - 1 - k0);
        if (!gated || stream_wait_value32()((CUstream)sw, (CUdeviceptr)(uintptr_t)(ctx->d_progress + b), gate,
                                            CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS)
            CUDA_TRY(cudaStreamWaitEvent(sw, ctx->ev_ov[1], 0));
        rc = p_disc->include_j2
                 ? launch_window<true>(1, ctx->d_x, ctx->d_u, ctx->d_tf, P, n_sats, K, n_sub_disc, tab, n_int, 0, ctx->d_status, sw, k0, kc)
                 : launch_window<false>(1, ctx->d_x, ctx->d_u, ctx->d_tf, P, n_sats, K, n_sub_disc, tab, n_int, 0, ctx->d_status, sw, k0, kc);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(ctx->ev[b], sw));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_copy, ctx->ev[b], 0));
        // the window's columns are one contiguous range per row: [k0 n_sats, (k0 + kc) n_sats)
        if ((rc = copy_out_chunk(out_host, ctx->d_out, n_int, (long long)k0 * n_sats, (long long)kc * n_sats, ctx->s_copy))) return rc;
    }
    // trajectory, inputs and status words follow the matrices on the copy stream (the propagation has long finished)
    CUDA_TRY(cudaStreamWaitEvent(ctx->s_copy, ctx->ev_ov[1], 0));
    if (y_host) CUDA_TRY(cudaMemcpyAsync(y_host, ctx->d_x, (size_t)n_sats * 7 * K * sizeof(double), cudaMemcpyDeviceToHost, ctx->s_copy));
    if (u_host) CUDA_TRY(cudaMemcpyAsync(u_host, ctx->d_u, (size_t)n_sats * 3 * K * sizeof(double), cudaMemcpyDeviceToHost, ctx->s_copy));
    fill_const_rows(out_host, n_int);
    if (status_host) {
        if ((rc = ensure_stage(ctx, (size_t)n_int + n_sats))) return rc;
        CUDA_TRY(cudaMemcpyAsync(is_pinned(status_host) ? status_host : ctx->h_stage, ctx->d_status, (size_t)n_int * sizeof(int32_t),
                                 cudaMemcpyDeviceToHost, ctx->s_copy));
        CUDA_TRY(cudaMemcpyAsync(ctx->h_stage + n_int, ctx->d_status2, (size_t)n_sats * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->s_copy));
    }
    CUDA_TRY(cudaStreamSynchronize(ctx->s_copy));
    CUDA_TRY(cudaStreamSynchronize(ctx->s_prop));
    for (cudaStream_t w : ctx->s_win) CUDA_TRY(cudaStreamSynchronize(w));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (status_host) {
        if (!is_pinned(status_host)) memcpy(status_host, ctx->h_stage, (size_t)n_int * sizeof(int32_t));
        const int32_t *ps = ctx->h_stage + n_int;
        for (int s = 0; s < n_sats; ++s)
            if (ps[s])
                for (int k = 0; k < K - 1; ++k) status_host[(size_t)s * (K - 1) + k] = ps[s];
    }
    return MPC_SUCCESS;
}

extern "C" int mpc_propagate_discretize(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                                        const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T,
                                        int n_sub_prop, int n_sub_disc, double *x, double *u, double *out,
                                        int64_t out_pitch, int64_t out_offset, int32_t *status_prop,
                                        int32_t *status_disc, int n_windows, void *stream)
{
    if (!out) return fail(MPC_E_INVALID, "null pointer argument");
    double *dst[1] = {out};
    return prop_disc_overlapped(ctx, y0, tf, p_prop, p_disc, ctrl, n_sats, T, n_sub_prop, n_sub_disc, x, u, dst, 1,
                                out_pitch, out_offset, status_prop, status_disc, n_windows, (cudaStream_t)stream);
}

extern "C" int mpc_propagate_discretize_multi(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                                              const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T,
                                              int n_sub_prop, int n_sub_disc, double *x, double *u, double *const *dst,
                                              int n_dst, int64_t out_pitch, int64_t out_offset, int32_t *status_prop,
                                              int32_t *status_disc, int n_windows, void *stream)
{
    return prop_disc_overlapped(ctx, y0, tf, p_prop, p_disc, ctrl, n_sats, T, n_sub_prop, n_sub_disc, x, u, dst, n_dst,
                                out_pitch, out_offset, status_prop, status_disc, n_windows, (cudaStream_t)stream);
}

namespace {

int gather_call(const mpc_gather_opts *g, int n_sats, int K, GatherCall &gc, int64_t &pitch, int64_t &offset)
{
    if (!g) return fail(MPC_E_INVALID, "null gather options");
    if (g->layout != MPC_LAYOUT_SAT_MAJOR && g->layout != MPC_LAYOUT_K_MAJOR) return fail(MPC_E_INVALID, "unknown layout %d", g->layout);
    if (g->skip_const < 0 || g->skip_const > 2 || g->stagger_phases < 0 || g->stagger_phases > 64)
        return fail(MPC_E_INVALID, "bad gather options (%d, %d)", g->skip_const, g->stagger_phases);
    if (g->sat_offset < 0 || g->n_sats_total < g->sat_offset + n_sats)
        return fail(MPC_E_INVALID, "n_sats_total / sat_offset do not hold this rank's satellites");
    gc.active = true;
    gc.skip_const = g->skip_const;
    gc.stagger = g->stagger_phases;
    gc.km_ntot = (g->layout == MPC_LAYOUT_K_MAJOR) ? g->n_sats_total : 0;
    gc.km_soff = (g->layout == MPC_LAYOUT_K_MAJOR) ? g->sat_offset : 0;
    pitch = g->n_sats_total * (int64_t)(K - 1);
    offset = g->sat_offset * (int64_t)(K - 1);
    return MPC_SUCCESS;
}

}  // namespace

extern "C" int mpc_discretize_batch_gather(const double *x, const double *u, const double *tf, const mpc_params *p,
                                           int n_sats, int K, int n_sub, double *const *dst, int n_dst,
                                           const mpc_gather_opts *g, int32_t *status, void *stream)
{
    if (K < 2) return fail(MPC_E_INVALID, "need K >= 2");
    GatherCall gc;
    int64_t pitch = 0, offset = 0;
    int rc = gather_call(g, n_sats, K, gc, pitch, offset);
    if (rc) return rc;
    GatherScope scope(gc);
    return disc_device(x, u, tf, p, n_sats, K, n_sub, dst, n_dst, pitch, offset, status, (cudaStream_t)stream);
}

extern "C" int mpc_propagate_discretize_gather(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                                               const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T,
                                               int n_sub_prop, int n_sub_disc, double *x, double *u, double *const *dst,
                                               int n_dst, const mpc_gather_opts *g, int32_t *status_prop,
                                               int32_t *status_disc, int n_windows, void *stream)
{
    if (T < 2) return fail(MPC_E_INVALID, "need T >= 2");
    GatherCall gc;
    int64_t pitch = 0, offset = 0;
    int rc = gather_call(g, n_sats, T, gc, pitch, offset);
    if (rc) return rc;
    GatherScope scope(gc);
    return prop_disc_overlapped(ctx, y0, tf, p_prop, p_disc, ctrl, n_sats, T, n_sub_prop, n_sub_disc, x, u, dst, n_dst, pitch,
                                offset, status_prop, status_disc, n_windows, (cudaStream_t)stream);
}

extern "C" {

// ------------------------------------------------------------------------------------- copy-engine gather
int mpc_fill_const_rows(double *out, int64_t out_pitch, void *stream)
{
    if (!out || out_pitch < 0) return fail(MPC_E_INVALID, "bad argument");
    if (out_pitch == 0) return MPC_SUCCESS;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(out + (size_t)kConstRow0 * out_pitch, 0, (size_t)6 * out_pitch * sizeof(double), st));
    const unsigned grid = (unsigned)std::min<long long>((out_pitch + 255) / 256, 148LL * 8);
    mpc::fill_kernel<<<grid, 256, 0, st>>>(out + (size_t)(kConstRow1 - 1) * out_pitch, (long long)out_pitch, 1.0);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

int mpc_discretize_batch_push(mpc_ctx *ctx, const double *x, const double *u, const double *tf, const mpc_params *p,
                              int n_sats, int K, int n_sub, double *const *dst, int n_dst, int64_t out_pitch,
                              int64_t out_offset, int32_t *status, int chunk_waves, int use_copy_kernel, void *stream)
{
    if (!ctx) return fail(MPC_E_INVALID, "null ctx");
    int rc = check_disc_args(x, u, tf, p, n_sats, K, n_sub);
    if (rc) return rc;
    if (p->include_drag) return fail(MPC_E_UNSUPPORTED, "include_drag is not supported by the push gather");
    if (!dst || n_dst < 1 || n_dst > MPC_MAX_DST) return fail(MPC_E_INVALID, "bad destination list");
    for (int d = 0; d < n_dst; ++d)
        if (!dst[d]) return fail(MPC_E_INVALID, "null destination %d", d);
    const long long n_int = (long long)n_sats * (K - 1);
    if (out_pitch < out_offset + n_int || out_offset < 0) return fail(MPC_E_INVALID, "out_pitch/out_offset do not hold the batch");
    if (n_int == 0) return MPC_SUCCESS;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    for (int d = 1; d < n_dst; ++d)
        if (!ctx->s_push[d]) CUDA_TRY(cudaStreamCreateWithFlags(&ctx->s_push[d], cudaStreamNonBlocking));
    if (use_copy_kernel && !ctx->s_pushk) {
        // the copy kernels must get SM slots ahead of the compute CTAs still queued: highest stream priority
        int lo = 0, hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&ctx->s_pushk, cudaStreamNonBlocking, hi));
    }
    mpc::PeerTab peers{};
    for (int d = 1; d < n_dst; ++d) peers.p[d - 1] = dst[d];
    const int cs = (int)std::min<long long>((long long)chunk_sats(ctx, n_sats, K) * std::max(chunk_waves, 1), n_sats);
    const int n_chunks = (n_sats + cs - 1) / cs;
    for (cudaStream_t &a : ctx->s_aux)
        if (!a) CUDA_TRY(cudaStreamCreateWithFlags(&a, cudaStreamNonBlocking));
    while (ctx->ev_push.size() < (size_t)n_chunks + MPC_MAX_DST + 4) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->ev_push.push_back(e);
    }
    const mpc::DiscParams P = disc_params(p);
    mpc::DstTab tab{};
    tab.p[0] = dst[0];
    const size_t pitch_b = (size_t)out_pitch * sizeof(double);
    // The chunk kernels are independent: they rotate over three compute streams forked from the caller's stream,
    // so the CTAs of chunk c+1 fill the SMs while the last CTAs of chunk c drain (no bubble between chunks).
    const size_t ev_fork = (size_t)n_chunks + MPC_MAX_DST;
    CUDA_TRY(cudaEventRecord(ctx->ev_push[ev_fork], st));
    for (cudaStream_t a : ctx->s_aux) CUDA_TRY(cudaStreamWaitEvent(a, ctx->ev_push[ev_fork], 0));
    for (int c = 0; c < n_chunks; ++c) {
        const int s0 = c * cs, ns = std::min(cs, n_sats - s0);
        const long long off = out_offset + (long long)s0 * (K - 1), nc = (long long)ns * (K - 1);
        const double *dx = x + (size_t)s0 * 7 * K, *du = u + (size_t)s0 * 3 * K;
        int32_t *stc = status ? status + (size_t)s0 * (K - 1) : nullptr;
        cudaStream_t sk = ctx->s_aux[c % 3];
        rc = p->include_j2 ? launch_disc_n<true, 1>(dx, du, tf + s0, P, ns, K, n_sub, tab, out_pitch, off, stc, sk)
                           : launch_disc_n<false, 1>(dx, du, tf + s0, P, ns, K, n_sub, tab, out_pitch, off, stc, sk);
        if (rc) return rc;
        if (n_dst == 1) continue;
        CUDA_TRY(cudaEventRecord(ctx->ev_push[c], sk));
        if (use_copy_kernel) {
            CUDA_TRY(cudaStreamWaitEvent(ctx->s_pushk, ctx->ev_push[c], 0));
            mpc::push_chunk_kernel<<<(unsigned)ctx->sm_count, 256, 0, ctx->s_pushk>>>(dst[0], peers, n_dst - 1, out_pitch, off, nc);
            g_launches.fetch_add(1, std::memory_order_relaxed);
            CUDA_TRY(cudaGetLastError());
            continue;
        }
        // peers in rotated order per chunk so that the copy engines do not all target the same GPU at once
        for (int i = 1; i < n_dst; ++i) {
            const int d = 1 + (i - 1 + c) % (n_dst - 1);
            cudaStream_t ps = ctx->s_push[d];
            CUDA_TRY(cudaStreamWaitEvent(ps, ctx->ev_push[c], 0));
            CUDA_TRY(cudaMemcpy2DAsync(dst[d] + off, pitch_b, dst[0] + off, pitch_b, (size_t)nc * sizeof(double), kConstRow0,
                                       cudaMemcpyDeviceToDevice, ps));
            CUDA_TRY(cudaMemcpy2DAsync(dst[d] + (size_t)kConstRow1 * out_pitch + off, pitch_b,
                                       dst[0] + (size_t)kConstRow1 * out_pitch + off, pitch_b, (size_t)nc * sizeof(double),
                                       MPC_OUT_ROWS - kConstRow1, cudaMemcpyDeviceToDevice, ps));
        }
    }
    for (int d = 1; d < n_dst; ++d) {   // the caller's stream continues only when every push has landed
        cudaStream_t ps = use_copy_kernel ? ctx->s_pushk : ctx->s_push[d];
        CUDA_TRY(cudaEventRecord(ctx->ev_push[(size_t)n_chunks + d], ps));
        CUDA_TRY(cudaStreamWaitEvent(st, ctx->ev_push[(size_t)n_chunks + d], 0));
        if (use_copy_kernel) break;
    }
    for (int a = 0; a < 3; ++a) {       // ... and every chunk kernel has finished
        CUDA_TRY(cudaEventRecord(ctx->ev_push[ev_fork + 1 + a], ctx->s_aux[a]));
        CUDA_TRY(cudaStreamWaitEvent(st, ctx->ev_push[ev_fork + 1 + a], 0));
    }
    return MPC_SUCCESS;
}

// ---------------------------------------------------------------------------------------------- constraint terms
static int cterms_check(const void *x, const void *u, int n_sats, int K, int Ku, const void *rbar, const void *ubar,
                        const void *fin)
{
    if (!x || !u || !rbar || !ubar || !fin) return fail(MPC_E_INVALID, "null pointer argument");
    if (n_sats < 0 || K < 2 || Ku < 1) return fail(MPC_E_INVALID, "need n_sats >= 0, K >= 2, Ku >= 1 (got %d, %d, %d)", n_sats, K, Ku);
    return MPC_SUCCESS;
}

static int cterms_launch(const double *x, const double *u, int n_sats, int K, int Ku, double mu, double *rbar,
                         double *ubar, double *fin, cudaStream_t st)
{
    const long long n = (long long)n_sats * std::max(K, Ku);
    const unsigned grid = (unsigned)((n + 255) / 256);
    mpc::constraint_terms_kernel<<<grid, 256, 0, st>>>(x, u, n_sats, K, Ku, mu, 2.220446049250313e-16, rbar, ubar, fin);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

int mpc_constraint_terms(const double *x, const double *u, int n_sats, int K, int u_cols, double mu, double *rbar_hat,
                         double *ubar_hat, double *final_terms, void *stream)
{
    int rc = cterms_check(x, u, n_sats, K, u_cols, rbar_hat, ubar_hat, final_terms);
    if (rc || n_sats == 0) return rc;
    return cterms_launch(x, u, n_sats, K, u_cols, mu, rbar_hat, ubar_hat, final_terms, (cudaStream_t)stream);
}

int mpc_constraint_terms_host(mpc_ctx *ctx, const double *x, const double *u, int n_sats, int K, int u_cols, double mu,
                              double *rbar_hat, double *ubar_hat, double *final_terms)
{
    if (!ctx) return fail(MPC_E_INVALID, "null ctx");
    int rc = cterms_check(x, u, n_sats, K, u_cols, rbar_hat, ubar_hat, final_terms);
    if (rc || n_sats == 0) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const size_t nx = (size_t)n_sats * 7 * K, nu = (size_t)n_sats * 3 * u_cols, nr = (size_t)n_sats * 3 * (K - 1),
                 nf = (size_t)n_sats * MPC_FINAL_TERMS;
    if ((rc = ensure(ctx->d_x, ctx->cap_x, nx))) return rc;
    if ((rc = ensure(ctx->d_u, ctx->cap_u, nu))) return rc;
    if ((rc = ensure(ctx->d_out, ctx->cap_out, nr + nu + nf))) return rc;
    cudaStream_t st = ctx->s_compute;
    double *d_r = ctx->d_out, *d_ub = d_r + nr, *d_f = d_ub + nu;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_x, x, nx * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_u, u, nu * sizeof(double), cudaMemcpyHostToDevice, st));
    if ((rc = cterms_launch(ctx->d_x, ctx->d_u, n_sats, K, u_cols, mu, d_r, d_ub, d_f, st))) return rc;
    CUDA_TRY(cudaMemcpyAsync(rbar_hat, d_r, nr * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(ubar_hat, d_ub, nu * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(final_terms, d_f, nf * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return MPC_SUCCESS;
}

int mpc_dynamics_jacobian(const double *soa, int64_t pitch, int64_t offset, int n_sats, int K, double *values,
                          int64_t *indices, double *rhs, void *stream)
{
    if (!soa || !values || !rhs) return fail(MPC_E_INVALID, "null pointer argument");
    if (n_sats < 0 || K < 2) return fail(MPC_E_INVALID, "need n_sats >= 0, K >= 2");
    const long long rows = (long long)n_sats * 7 * (K - 1);
    if (pitch < offset + (long long)n_sats * (K - 1) || offset < 0) return fail(MPC_E_INVALID, "pitch/offset do not hold the batch");
    if (rows == 0) return MPC_SUCCESS;
    const unsigned grid = (unsigned)((rows + 255) / 256);
    mpc::dynamics_jacobian_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(soa, pitch, offset, n_sats, K, values, indices, rhs);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

// ---- ragged batches (satellite s on K_s nodes, buffers padded to K_max): one launch over the live intervals ----------
static int cterms_ragged_launch(const double *x, const double *u, int n_sats, int K_max, long long n_live,
                                const long long *first, double mu, double *rbar, double *ubar, double *fin, cudaStream_t st)
{
    const unsigned grid = (unsigned)((n_live + 255) / 256);
    mpc::constraint_terms_kernel<true><<<grid, 256, 0, st>>>(x, u, n_sats, K_max, K_max, mu, 2.220446049250313e-16, rbar, ubar,
                                                             fin, first);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

int mpc_constraint_terms_ragged(const double *x, const double *u, int n_sats, int K_max, const int32_t *K_sat, int64_t *first,
                                double mu, double *rbar_hat, double *ubar_hat, double *final_terms, void *stream)
{
    int rc = cterms_check(x, u, n_sats, K_max, K_max, rbar_hat, ubar_hat, final_terms);
    if (rc || (rc = check_counts(K_sat, n_sats, K_max, "K_sat"))) return rc;
    if (!first) return fail(MPC_E_INVALID, "null first");
    if (n_sats == 0) return MPC_SUCCESS;
    cudaStream_t st = (cudaStream_t)stream;
    const std::vector<long long> f = ragged_first(K_sat, n_sats);
    CUDA_TRY(cudaMemcpyAsync(first, f.data(), f.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    return cterms_ragged_launch(x, u, n_sats, K_max, f[n_sats], (const long long *)first, mu, rbar_hat, ubar_hat, final_terms, st);
}

int mpc_constraint_terms_ragged_host(mpc_ctx *ctx, const double *x, const double *u, int n_sats, int K_max,
                                     const int32_t *K_sat, double mu, double *rbar_hat, double *ubar_hat, double *final_terms)
{
    if (!ctx) return fail(MPC_E_INVALID, "null ctx");
    int rc = cterms_check(x, u, n_sats, K_max, K_max, rbar_hat, ubar_hat, final_terms);
    if (rc || (rc = check_counts(K_sat, n_sats, K_max, "K_sat")) || n_sats == 0) return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const size_t nx = (size_t)n_sats * 7 * K_max, nu = (size_t)n_sats * 3 * K_max, nr = (size_t)n_sats * 3 * (K_max - 1),
                 nf = (size_t)n_sats * MPC_FINAL_TERMS;
    const std::vector<long long> f = ragged_first(K_sat, n_sats);
    if ((rc = ensure(ctx->d_x, ctx->cap_x, nx))) return rc;
    if ((rc = ensure(ctx->d_u, ctx->cap_u, nu))) return rc;
    if ((rc = ensure(ctx->d_out, ctx->cap_out, nr + nu + nf))) return rc;
    if ((rc = ensure(ctx->d_first, ctx->cap_first, f.size()))) return rc;
    cudaStream_t st = ctx->s_compute;
    double *d_r = ctx->d_out, *d_ub = d_r + nr, *d_f = d_ub + nu;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_x, x, nx * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_u, u, nu * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_first, f.data(), f.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    // the kernel leaves the padding columns alone: they go back as NaN (all-ones bytes)
    CUDA_TRY(cudaMemsetAsync(d_r, 0xFF, (nr + nu) * sizeof(double), st));
    if ((rc = cterms_ragged_launch(ctx->d_x, ctx->d_u, n_sats, K_max, f[n_sats], ctx->d_first, mu, d_r, d_ub, d_f, st))) return rc;
    CUDA_TRY(cudaMemcpyAsync(rbar_hat, d_r, nr * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(ubar_hat, d_ub, nu * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(final_terms, d_f, nf * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return MPC_SUCCESS;
}

int mpc_dynamics_jacobian_ragged(const double *soa, int64_t pitch, int64_t offset, int n_sats, int K_max,
                                 const int32_t *K_sat, int64_t *first, double *values, int64_t *indices, double *rhs,
                                 void *stream)
{
    if (!soa || !values || !rhs || !first) return fail(MPC_E_INVALID, "null pointer argument");
    if (n_sats < 0 || K_max < 2) return fail(MPC_E_INVALID, "need n_sats >= 0, K_max >= 2 (got %d, %d)", n_sats, K_max);
    if (pitch < offset + (long long)n_sats * (K_max - 1) || offset < 0) return fail(MPC_E_INVALID, "pitch/offset do not hold the batch");
    int rc = check_counts(K_sat, n_sats, K_max, "K_sat");
    if (rc || n_sats == 0) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const std::vector<long long> f = ragged_first(K_sat, n_sats);
    CUDA_TRY(cudaMemcpyAsync(first, f.data(), f.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    const unsigned grid = (unsigned)((f[n_sats] + 255) / 256);
    mpc::dynamics_jacobian_kernel<true><<<grid, 256, 0, st>>>(soa, pitch, offset, n_sats, K_max, values, indices, rhs,
                                                              (const long long *)first);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return MPC_SUCCESS;
}

// ---- per-satellite designer units: MU of every satellite from its own constants ----------------------------------------
static int cterms_units_launch(const double *x, const double *u, int n_sats, int K_max, long long n_units, const long long *first,
                               const double *mu_sat, double *rbar, double *ubar, double *fin, cudaStream_t st)
{
    if (mpc_units_sizeof(0) != sizeof(mpc::DiscParams)) return fail(MPC_E_CUDA, "mpc_b200_units.cu was built against different parameter structs");
    CUDA_TRY(mpc_units_launch_cterms(x, u, n_sats, K_max, n_units, first, mu_sat, rbar, ubar, fin, st));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return MPC_SUCCESS;
}

static std::vector<double> mu_table(const mpc_sat_consts *c, int n)
{
    std::vector<double> v((size_t)n);
    for (int s = 0; s < n; ++s) v[s] = c[s].mu;
    return v;
}

int mpc_constraint_terms_units(const double *x, const double *u, int n_sats, int K_max, const int32_t *K_sat, int64_t *first,
                               const mpc_sat_consts *consts, double *consts_scratch, double *rbar_hat, double *ubar_hat,
                               double *final_terms, void *stream)
{
    int rc = cterms_check(x, u, n_sats, K_max, K_max, rbar_hat, ubar_hat, final_terms);
    if (rc || (K_sat && (rc = check_counts(K_sat, n_sats, K_max, "K_sat"))) || (rc = check_sat_consts(consts, n_sats))) return rc;
    if ((K_sat && !first) || !consts_scratch) return fail(MPC_E_INVALID, "null first / consts_scratch");
    if (n_sats == 0) return MPC_SUCCESS;
    cudaStream_t st = (cudaStream_t)stream;
    const std::vector<double> mu = mu_table(consts, n_sats);
    CUDA_TRY(cudaMemcpyAsync(consts_scratch, mu.data(), mu.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    long long n_units = (long long)n_sats * K_max;
    if (K_sat) {
        const std::vector<long long> f = ragged_first(K_sat, n_sats);
        CUDA_TRY(cudaMemcpyAsync(first, f.data(), f.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
        n_units = f[n_sats];
    }
    return cterms_units_launch(x, u, n_sats, K_max, n_units, K_sat ? (const long long *)first : nullptr, consts_scratch, rbar_hat,
                               ubar_hat, final_terms, st);
}

int mpc_constraint_terms_units_host(mpc_ctx *ctx, const double *x, const double *u, int n_sats, int K_max,
                                    const int32_t *K_sat, const mpc_sat_consts *consts, double *rbar_hat, double *ubar_hat,
                                    double *final_terms)
{
    if (!ctx) return fail(MPC_E_INVALID, "null ctx");
    int rc = cterms_check(x, u, n_sats, K_max, K_max, rbar_hat, ubar_hat, final_terms);
    if (rc || (K_sat && (rc = check_counts(K_sat, n_sats, K_max, "K_sat"))) || (rc = check_sat_consts(consts, n_sats)) || n_sats == 0)
        return rc;
    CUDA_TRY(cudaSetDevice(ctx->device));
    const size_t nx = (size_t)n_sats * 7 * K_max, nu = (size_t)n_sats * 3 * K_max, nr = (size_t)n_sats * 3 * (K_max - 1),
                 nf = (size_t)n_sats * MPC_FINAL_TERMS;
    if ((rc = ensure(ctx->d_x, ctx->cap_x, nx))) return rc;
    if ((rc = ensure(ctx->d_u, ctx->cap_u, nu))) return rc;
    if ((rc = ensure(ctx->d_out, ctx->cap_out, nr + nu + nf))) return rc;
    if ((rc = ensure(ctx->d_psc, ctx->cap_psc, (size_t)n_sats * MPC_SAT_SCRATCH_DOUBLES))) return rc;
    cudaStream_t st = ctx->s_compute;
    double *d_r = ctx->d_out, *d_ub = d_r + nr, *d_f = d_ub + nu;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_x, x, nx * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_u, u, nu * sizeof(double), cudaMemcpyHostToDevice, st));
    const std::vector<double> mu = mu_table(consts, n_sats);
    CUDA_TRY(cudaMemcpyAsync(ctx->d_psc, mu.data(), mu.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    long long n_units = (long long)n_sats * K_max;
    if (K_sat) {
        const std::vector<long long> f = ragged_first(K_sat, n_sats);
        if ((rc = ensure(ctx->d_first, ctx->cap_first, f.size()))) return rc;
        CUDA_TRY(cudaMemcpyAsync(ctx->d_first, f.data(), f.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
        n_units = f[n_sats];
        // the kernel leaves the padding columns alone: they go back as NaN (all-ones bytes)
        CUDA_TRY(cudaMemsetAsync(d_r, 0xFF, (nr + nu) * sizeof(double), st));
    }
    if ((rc = cterms_units_launch(ctx->d_x, ctx->d_u, n_sats, K_max, n_units, K_sat ? ctx->d_first : nullptr, ctx->d_psc, d_r, d_ub,
                                  d_f, st)))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(rbar_hat, d_r, nr * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(ubar_hat, d_ub, nu * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(final_terms, d_f, nf * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return MPC_SUCCESS;
}

int mpc_fp64_peak_probe(int device, int repeats, double *tflops, double *ms)
{
    if (!tflops) return fail(MPC_E_INVALID, "null output");
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    double *d = nullptr;
    CUDA_TRY(cudaMalloc((void **)&d, (size_t)blocks * threads * sizeof(double)));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int r = 0; r < std::max(repeats, 1) + 1; ++r) {
        CUDA_TRY(cudaEventRecord(e0, 0));
        mpc::fp64_probe_kernel<<<blocks, threads>>>(d, iters, 1.0 + r);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        CUDA_TRY(cudaEventRecord(e1, 0));
        CUDA_TRY(cudaEventSynchronize(e1));
        float t = 0;
        CUDA_TRY(cudaEventElapsedTime(&t, e0, e1));
        if (r > 0) best = std::min(best, t);  // first launch is warm-up
    }
    CUDA_TRY(cudaGetLastError());
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    const double flops = (double)blocks * threads * (double)iters * 64.0 * 2.0;
    *tflops = flops / (best * 1e-3) / 1e12;
    if (ms) *ms = best;
    return MPC_SUCCESS;
}

}  // extern "C"
