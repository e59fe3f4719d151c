// Fused FFJORD continuous-normalising-flow sweeps (BASELINE config 3).
//
// Reference path replaced: per stage, PETSc calls evalRHSFunction (pnode/petsc_adjoint.py:393-412) -> FlattenFunc ->
// ODEfunc.forward (ffjord-pnode/lib/layers/odefunc.py:345-385), which runs the ConcatSquash MLP AND a torch.autograd.grad
// with create_graph=True for the Hutchinson trace (odefunc.py:53-57); per adjoint stage RHSJacShell.multTranspose
// (petsc_adjoint.py:52-82) re-evaluates all of that and differentiates THROUGH the inner autograd.grad (second order).
// Here both are closed-form per trajectory:
//     p_j = W1[j,:] z + b1_j      a_j = p_j g1_j(t) + c1_j(t)      s_j = softplus(a_j)      sg_j = sigmoid(a_j)
//     dz_k = (W2[k,:] s + b2_k) g2_k(t) + c2_k(t)
//     e^T J e = sum_j g1_j sg_j w_j q_j,   w_j = sum_k W2[k,j] g2_k e_k,   q_j = W1[j,:] e        (J = d dz / d z)
// with g = sigmoid(hgw t + hgb), c = hb t the ConcatSquash gates (diffeq_layers/basic.py:76-86).  Only sg_j depends on z
// inside the trace, which makes the VJP of the trace (the "second-order" part) one extra multiply-add per hidden unit.
//
// B200 mapping: CUDA-core kernels (D = 6, H = 60: GEMMs of K = 6 are not tensor-core shaped), one trajectory per thread,
// weights packed per hidden unit in SMEM and broadcast, gates of every stage time precomputed once per launch.
//  * cnf_rk_attempt_kernel: ONE launch = all stages of one step attempt + completion + embedded error + deterministic
//    weighted-squared-error reduction (device scalar; the caller all-reduces it across GPUs before accept/reject).
//  * cnf_rk_adj_kernel: ONE launch = the whole discrete-adjoint sweep.  Parameter gradients (984 scalars) are reduced with
//    the same warp-private transposed SMEM tile as csrc/mlp_rk.cu (lane = hidden unit in the reduce phase), layer-2 gate /
//    bias gradients in per-thread registers; per-block partials are combined in fixed order by the last block.
#include <mutex>
#include <string.h>

#include "common.cuh"
#include "f32x2.cuh"

// tuning parameters (tools/tune_cnf.py builds -D variants; the defaults are the measured best)
#ifndef CNF_P1_UNROLL
#define CNF_P1_UNROLL 2  // adjoint phase 1: hidden units in flight per thread
#endif
#ifndef CNF_P2_UNROLL
#define CNF_P2_UNROLL 2  // adjoint phase 2: 16-byte trajectory vectors in flight per lane
#endif
#ifndef CNF_ATT_MINB
#define CNF_ATT_MINB 2   // attempt kernel: CTAs per SM the register allocation aims at
#endif
#ifndef CNF_EVAL_UNROLL
#define CNF_EVAL_UNROLL 4  // attempt kernel: hidden units in flight per thread
#endif
#define CNF_PRAGMA_(x) _Pragma(#x)
#define CNF_UNROLL(n) CNF_PRAGMA_(unroll n)

namespace pnode {

template <typename T>
struct CnfPtrs {
    const T *w1, *b1, *hb1, *hgw1, *hgb1, *w2, *b2, *hb2, *hgw2, *hgb2, *e;
    int t_f32;
};

template <typename T, int D>
struct alignas(16) UnitC {
    T w1[D];  // W1[j][:]
    T w2[D];  // W2[:][j]
    T b1;
    T pad[3];
};

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ double sigmoid_acc(double x) { return 1.0 / (1.0 + exp(-x)); }

// softplus (torch.nn.Softplus: beta 1, threshold 20) and its derivative, from one exponential
// fp32: three MUFU ops (ex2, rcp, lg2); absolute error ~1e-7, far inside the 1e-4 parity bar of the fp32 path
__device__ __forceinline__ void softplus_sigmoid(float a, float &s, float &sg) {
    float E, r, l;
    const float x = -1.4426950408889634f * fabsf(a);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(E) : "f"(x));
    const float d = 1.0f + E;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(d));
    sg = a >= 0.0f ? r : E * r;
    // no threshold branch: for a > 20, E < 2^-28 so d rounds to 1, lg2(1) = +0 and s = a exactly, and rcp(1) = 1 so sg = 1
    // exactly -- the value, slope and zero curvature of torch's Softplus above its threshold
    s = fmaf(l, 0.6931471805599453f, fmaxf(a, 0.0f));
}
// two trajectories at once: the MUFU part is per half, the arithmetic around it packed
__device__ __forceinline__ void softplus_sigmoid(F2 a, F2 &s, F2 &sg) {
    float a0, a1, E0, E1, r0, r1, l0, l1, d0, d1;
    unpk(a, a0, a1);
    const float x0 = -1.4426950408889634f * fabsf(a0), x1 = -1.4426950408889634f * fabsf(a1);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(E0) : "f"(x0));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(E1) : "f"(x1));
    unpk(pk(E0, E1) + 1.0f, d0, d1);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(d0));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(d1));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l0) : "f"(d0));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l1) : "f"(d1));
    sg = pk(a0 >= 0.0f ? r0 : E0 * r0, a1 >= 0.0f ? r1 : E1 * r1);
    s = fma(pk(l0, l1), 0.6931471805599453f, pk(fmaxf(a0, 0.0f), fmaxf(a1, 0.0f)));
}
__device__ __forceinline__ void softplus_sigmoid(double a, double &s, double &sg) {
    // torch's threshold: above 20, E = 0 makes s = a and sg = 1 exactly -- the value, slope and zero curvature of the
    // identity (sigmoid(20) = 1 - 2e-9 would miss the fp64 parity bar), so the adjoint's 1 - sg is exactly 0
    const double E = a > 20.0 ? 0.0 : exp(-fabs(a));
    const double r = 1.0 / (1.0 + E);
    sg = a >= 0.0 ? r : E * r;
    s = fmax(a, 0.0) + log1p(E);
}

// shared-memory image of the model for one launch
template <typename T, int D, int H, int S>
struct CnfShared {
    UnitC<T, D> unit[H];
    T g1[S][H], c1[S][H];   // layer-1 gate / bias at every stage time
    T g2[S][D], c2[S][D];
    T b2[D];
    T tstage[S];
    T ha[S][S], hb[S], he[S];  // h a_ij, h b_j, h (be_j - b_j): the stage / completion / error coefficients of this step
    T adj_r[S][S], adj_c[S];   // adjoint stage recurrences (SURVEY.md A.4): a_ji / b_i and h b_i (a_ji and h where b_i = 0)
    int adj_has_b[S];
};

// Stage time as the module sees it.  FFJORD's ODEfunc does `t = torch.tensor(t).type_as(y)` (odefunc.py:356):
// torch.tensor(python float) is float32, so even a float64 run sees t rounded through fp32 (t_f32 != 0 reproduces that).
template <typename T>
__device__ __forceinline__ T stage_time(double t, int t_f32) {
    return t_f32 ? (T)(float)t : (T)t;
}

template <typename T, int D, int H, int S>
__device__ __forceinline__ void cnf_setup(CnfShared<T, D, H, S> &sm, const CnfPtrs<T> &w, const pnode_rk_tableau &tab,
                                          double t, double h) {
    for (int j = threadIdx.x; j < H; j += blockDim.x) {
        UnitC<T, D> u;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            u.w1[k] = w.w1[j * D + k];
            u.w2[k] = w.w2[k * H + j];
        }
        u.b1 = w.b1[j];
        u.pad[0] = u.pad[1] = u.pad[2] = T(0);
        sm.unit[j] = u;
        const T gw = w.hgw1[j], gb = w.hgb1[j], hb = w.hb1[j];
#pragma unroll
        for (int i = 0; i < S; ++i) {
            const T tt = stage_time<T>(t + tab.c[i] * h, w.t_f32);
            sm.g1[i][j] = sigmoid_acc(fma(gw, tt, gb));
            sm.c1[i][j] = hb * tt;
        }
    }
    if (threadIdx.x < D) {
        const int k = threadIdx.x;
        sm.b2[k] = w.b2[k];
        const T gw = w.hgw2[k], gb = w.hgb2[k], hb = w.hb2[k];
#pragma unroll
        for (int i = 0; i < S; ++i) {
            const T tt = stage_time<T>(t + tab.c[i] * h, w.t_f32);
            sm.g2[i][k] = sigmoid_acc(fma(gw, tt, gb));
            sm.c2[i][k] = hb * tt;
        }
    }
    if (threadIdx.x < S) {
        const int i = threadIdx.x;
        sm.tstage[i] = stage_time<T>(t + tab.c[i] * h, w.t_f32);
        sm.hb[i] = (T)(h * tab.b[i]);
        sm.he[i] = (T)(h * (tab.be[i] - tab.b[i]));
        const double bi = tab.b[i];
        sm.adj_has_b[i] = bi != 0.0;
        sm.adj_c[i] = (T)(bi != 0.0 ? h * bi : h);
#pragma unroll
        for (int j = 0; j < S; ++j) {
            sm.ha[i][j] = (T)(h * tab.a[i][j]);
            sm.adj_r[j][i] = (T)(bi != 0.0 ? tab.a[j][i] / bi : tab.a[j][i]);
        }
    }
}

// A trajectory slot may be spread over LPT adjacent lanes, each owning H / LPT hidden units (small batches: the dependent
// chain of one evaluation is LPT times shorter).  The partial sums over units are combined by an xor butterfly, which
// leaves bit-identical totals in all LPT lanes, so they carry identical copies of the state from then on.
__device__ __forceinline__ double shfl_x(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ F2 shfl_x(F2 v, int m) {
    F2 r;
    r.v = __shfl_xor_sync(0xffffffffu, v.v, m);
    return r;
}
template <int LPT, typename V>
__device__ __forceinline__ V sub_sum(V v) {
#pragma unroll
    for (int m = 1; m < LPT; m <<= 1) v = v + shfl_x(v, m);
    return v;
}

// f(t_i, (z, .)): out[0..D) = dz, out[D] = -e^T J e -- for the Pack<T>::W trajectories a thread carries (fp64: one, plain
// doubles; fp32: two, in the halves of packed registers, every operation an FFMA2 / FMUL2 / FADD2)
// qcol: the thread's column of q_j = W1[j,:] e (stride CNF_THREADS), which does not depend on the stage -- computed once
// per attempt by the caller.
template <typename T, int D, int H, int S, int LPT, typename V>
__device__ __forceinline__ void cnf_eval(const CnfShared<T, D, H, S> &sm, int i, const V (&z)[D], const V (&e)[D],
                                         V (&out)[D + 1], const V *__restrict__ qcol, int qstride, int sub) {
    static_assert(H % LPT == 0, "hidden units must split evenly over the lanes of a slot");
    V ge[D], r[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        ge[k] = sm.g2[i][k] * e[k];
        r[k] = Pack<T>::all(sub == 0 ? sm.b2[k] : T(0));
    }
    V div = Pack<T>::all(T(0));
    const int jbeg = sub * (H / LPT), jend = jbeg + H / LPT;
    CNF_UNROLL(CNF_EVAL_UNROLL)
    for (int j = jbeg; j < jend; ++j) {
        const UnitC<T, D> u = sm.unit[j];
        V p = Pack<T>::all(u.b1), w = Pack<T>::all(T(0));
#pragma unroll
        for (int k = 0; k < D; ++k) {
            p = fma(u.w1[k], z[k], p);
            w = fma(u.w2[k], ge[k], w);
        }
        const V q = qcol[j * qstride];
        const T g1 = sm.g1[i][j];
        const V a = fma(p, g1, sm.c1[i][j]);
        V s, sg;
        softplus_sigmoid(a, s, sg);
#pragma unroll
        for (int k = 0; k < D; ++k) r[k] = fma(u.w2[k], s, r[k]);
        div = fma(g1 * sg, w * q, div);
    }
#pragma unroll
    for (int k = 0; k < D; ++k) out[k] = fma(sub_sum<LPT>(r[k]), sm.g2[i][k], sm.c2[i][k]);
    out[D] = -sub_sum<LPT>(div);
}

// ---------------------------------------------------------------------------------------------------------------------
// one step attempt

constexpr int CNF_THREADS = 128;
constexpr int CNF_MAX_BLOCKS = 148 * 8;

struct CnfWrmsWork {
    unsigned int ticket;
    unsigned int pad[15];
    double partial[CNF_MAX_BLOCKS];
};

// ---- step controller on the device: pnode_b200/controller.py (adapt_basic, TimeLoop.report, TimeLoop._matchstep) restated
// in double precision; run by ONE thread of the last block of an attempt -------------------------------------------------
namespace ctl {
constexpr double SAFETY = 0.9, REJECT_SAFETY = 0.5, CLIP_LO = 0.1, CLIP_HI = 10.0, DT_MIN = 1e-20, DT_MAX = 1e50;
constexpr double MATCH_NEAR = 0.01, MATCH_HALF = 2.0, SPAN_RELTOL = 1e-6, SPAN_ABSTOL = 10 * 2.220446049250313e-16;
constexpr double SQRT_EPS = 1.4901161193847656e-08;

__device__ inline double matchstep(pnode_cnf_ctl &c, double t_new, double h, double h_next) {
    bool hit = false;
    double tmax;
    if (c.nspan > 0) {
        const int k = min(c.ctr, c.nspan - 1);
        if (fabs(t_new - c.span[k]) <= SPAN_RELTOL * h + SPAN_ABSTOL) {
            hit = true;
            tmax = (k + 1 < c.nspan) ? c.span[k + 1] : c.t_end;
        } else {
            tmax = c.span[k];
        }
    } else {
        tmax = c.t_end;
    }
    double out = h_next;
    const double tend = t_new + h_next, hmax = tmax - t_new;
    if (t_new < tmax) {
        if (tend > tmax) {
            out = hmax;
        } else if (tend < tmax) {
            if (h_next * MATCH_HALF > hmax) out = hmax / 2;
            if (h_next * (1.0 + MATCH_NEAR) > hmax) out = hmax;
        }
    }
    if (c.nspan > 0) {
        if (h != out && c.dt_span_cached == 0.0) c.dt_span_cached = h;
        if (h == out && c.dt_span_cached != 0.0 && hit) {
            out = c.dt_span_cached;
            c.dt_span_cached = 0.0;
        }
    }
    return out;
}

// one attempt's verdict: updates the control block for the next attempt
__device__ inline void report(pnode_cnf_ctl &c, double sumsq) {
    const double h = c.h, enorm = sqrt(sumsq / c.n_global);
    double safety = SAFETY;
    bool accept = true;
    if (enorm > 1.0) {
        if (!c.prev_ok) safety *= REJECT_SAFETY;
        accept = h < (1.0 + SQRT_EPS) * DT_MIN;
    }
    double fac = enorm > 0.0 ? safety * pow(enorm, -1.0 / (double)c.order) : CLIP_HI;
    fac = fmin(fmax(fac, CLIP_LO), CLIP_HI);
    double h_next = fmin(fmax(h * fac, DT_MIN), DT_MAX);
    const int a = c.attempts;
    if (a < PNODE_CTL_MAX_LOG) {
        c.log_t[a] = c.t, c.log_h[a] = h, c.log_enorm[a] = enorm, c.log_accepted[a] = accept ? 1 : 0;
    }
    c.attempts = a + 1;
    if (!accept) {
        c.h = h_next;
        c.prev_ok = 0;
        c.rejections += 1;
        if (c.rejections > c.max_reject) c.done = 2;
    } else {
        const double t_old = c.t, t_new = c.t + h;
        h_next = matchstep(c, t_new, h, h_next);
        c.prev_ok = 1;
        c.rejections = 0;
        c.t = t_new;
        c.steps += 1;
        c.h = h_next;
        if (c.nspan > 0 && c.cur_sol_index < c.nspan && fabs(t_new - c.span[c.cur_sol_index]) < c.delta) c.cur_sol_index += 1;
        int slot = -1;
        if (c.nspan > 0 && c.ctr < c.nspan && fabs(t_new - c.span[c.ctr]) <= SPAN_RELTOL * h + SPAN_ABSTOL) slot = c.ctr++;
        c.pending_slot = slot;
        const int idx = c.steps - 1;  // this step, as the adjoint sweep will read it
        if (idx < PNODE_CTL_MAX_LOG) {
            c.sched[idx].t = t_old, c.sched[idx].h = h, c.sched[idx].out_slot = slot;
            c.sched[idx].in_slot = c.single ? -1 : (idx == 0 ? 0 : c.prev_out_slot);
        }
        c.prev_out_slot = slot;
        c.cur ^= 1;       // the candidate becomes the state
        c.kcur ^= 1;      // and its last stage slope the carried-over one
        c.have_k = 1;
        if (!(c.t < c.t_end && fabs(c.t - c.t_end) > SPAN_ABSTOL))
            c.done = 1;
        else if (c.max_steps > 0 && c.steps >= c.max_steps)
            c.done = 4;
    }
    if (c.attempts >= PNODE_CTL_MAX_LOG && c.done == 0) c.done = 3;
}
}  // namespace ctl

template <typename T, int D, int H, int S, int LPT>
__global__ void __launch_bounds__(CNF_THREADS, CNF_ATT_MINB)
cnf_rk_attempt_kernel(const CnfPtrs<T> w, const pnode_rk_tableau tab, const T *__restrict__ u,
                      const T *__restrict__ kfsal_in, const int64_t ntraj, double t, double h,
                      T *__restrict__ unew, T *__restrict__ kfsal_out, T *__restrict__ ckpt, const double atol,
                      const double rtol, double *__restrict__ sumsq, CnfWrmsWork *__restrict__ work,
                      pnode_cnf_ctl *__restrict__ dctl, T *__restrict__ ubuf, T *__restrict__ kbuf,
                      const int64_t ckpt_step_elems, T *__restrict__ sol, const unsigned long long loop_cond,
                      const PeerComm pc) {
    typedef Pack<T> P;
    typedef typename P::V V;
    constexpr int W = P::W;  // trajectories per thread
    T *sol_out = nullptr;
    if (dctl != nullptr) {
        // device-controlled attempt: time, step and buffers come from the control block the previous attempt's last block
        // wrote (every block reads it before any block of THIS launch can modify it: the update happens behind the ticket)
        const volatile pnode_cnf_ctl *vc = dctl;
        if (vc->done != 0) {
            // the WHILE node runs its body once per launch whatever the state: end the loop
            if (loop_cond != 0ull && blockIdx.x == 0 && threadIdx.x == 0) cudaGraphSetConditional(loop_cond, 0u);
            return;
        }
        t = vc->t, h = vc->h;
        const int64_t n = ntraj * (D + 1);
        const int cur = vc->cur, kcur = vc->kcur;
        u = ubuf + (int64_t)cur * n;
        unew = ubuf + (int64_t)(cur ^ 1) * n;
        kfsal_in = (tab.fsal && vc->have_k) ? kbuf + (int64_t)kcur * n : nullptr;
        kfsal_out = tab.fsal ? kbuf + (int64_t)(kcur ^ 1) * n : nullptr;
        if (ckpt != nullptr) ckpt += (int64_t)vc->steps * ckpt_step_elems;
        const int slot = vc->pending_slot;
        if (slot >= 0 && sol != nullptr) sol_out = sol + (int64_t)slot * n;
    }
    __shared__ CnfShared<T, D, H, S> sm;
    extern __shared__ __align__(16) unsigned char cnf_dyn_smem[];
    V *qcol = reinterpret_cast<V *>(cnf_dyn_smem) + threadIdx.x;  // [H][CNF_THREADS], this thread's column
    cnf_setup<T, D, H, S>(sm, w, tab, t, h);
    __syncthreads();
    constexpr int N = D + 1;
    const int s_eff = tab.fsal ? S - 1 : S;
    double local = 0.0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x / LPT;
    const int64_t nslots = (ntraj + W - 1) / W;
    const int sub = threadIdx.x % LPT;  // which share of the hidden units this lane owns
    // the trip count is uniform over a warp (the butterfly sums need all its lanes); slots past the end compute on zeros
    const int64_t wslot = ((int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31)) / LPT;
    const int64_t myslot = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPT;
    for (int64_t it = 0; wslot + it * stride < nslots; ++it) {
        const int64_t slot = myslot + it * stride;
        // trajectories tr[0..W) of this thread; a missing one (odd ntraj, tail of the warp) computes on zeros and stores nothing
        int64_t tr[W];
        bool ok[W], st[W];
#pragma unroll
        for (int x = 0; x < W; ++x) {
            tr[x] = slot * W + x;
            ok[x] = tr[x] < ntraj;
            st[x] = ok[x] && sub == 0;  // one lane of the slot stores
            if (!ok[x]) tr[x] = ntraj - 1;
        }
        auto gather = [&](const T *base, int64_t mul, int64_t off) -> V {
            T v[2] = {T(0), T(0)};
#pragma unroll
            for (int x = 0; x < W; ++x) v[x] = ok[x] ? base[tr[x] * mul + off] : T(0);
            return P::make(v[0], v[1]);
        };
        auto scatter = [&](T *base, int64_t mul, int64_t off, V val) {
#pragma unroll
            for (int x = 0; x < W; ++x)
                if (st[x]) base[tr[x] * mul + off] = P::get(val, x);
        };
        V y[N], e[D], K[S][N];
#pragma unroll
        for (int k = 0; k < D; ++k) {
            y[k] = gather(u, D, k);
            e[k] = gather(w.e, D, k);
        }
        y[D] = gather(u, 1, ntraj * D);
        // q_j = W1[j,:] e does not depend on the stage: once per attempt, into the thread's shared-memory column
#pragma unroll 4
        for (int j = sub * (H / LPT); j < (sub + 1) * (H / LPT); ++j) {
            V q = P::all(T(0));
#pragma unroll
            for (int k = 0; k < D; ++k) q = fma(sm.unit[j].w1[k], e[k], q);
            qcol[j * CNF_THREADS] = q;
        }
        if (sol_out != nullptr) {  // the state this attempt starts from landed on an output time
#pragma unroll
            for (int k = 0; k < D; ++k) scatter(sol_out, D, k, y[k]);
            scatter(sol_out, 1, ntraj * D, y[D]);
        }
        // the stage loop is NOT unrolled: the slopes K live in a small local array (touched ~50 times per stage, against
        // ~3000 instructions of right-hand side), which keeps the kernel at ~1/7 of the unrolled code size and registers
#pragma unroll 1
        for (int i = 0; i < S; ++i) {
            V Y[N];
#pragma unroll
            for (int k = 0; k < N; ++k) Y[k] = y[k];
            for (int j = 0; j < i; ++j) {
                const T ha = sm.ha[i][j];
#pragma unroll
                for (int k = 0; k < N; ++k) Y[k] = fma(ha, K[j][k], Y[k]);
            }
            if (ckpt != nullptr && i < s_eff) {
#pragma unroll
                for (int k = 0; k < D; ++k) scatter(ckpt, 1, ((int64_t)i * D + k) * ntraj, Y[k]);
            }
            if (i == 0 && kfsal_in != nullptr) {
#pragma unroll
                for (int k = 0; k < D; ++k) K[0][k] = gather(kfsal_in, D, k);
                K[0][D] = gather(kfsal_in, 1, ntraj * D);
            } else {
                V z[D];
#pragma unroll
                for (int k = 0; k < D; ++k) z[k] = Y[k];
                cnf_eval<T, D, H, S, LPT, V>(sm, i, z, e, K[i], qcol, CNF_THREADS, sub);
            }
        }
        V yn[N], err[N];
#pragma unroll
        for (int k = 0; k < N; ++k) {
            yn[k] = y[k];
            err[k] = P::all(T(0));
        }
        for (int j = 0; j < S; ++j) {
            const T hb = sm.hb[j], he = sm.he[j];
#pragma unroll
            for (int k = 0; k < N; ++k) {
                yn[k] = fma(hb, K[j][k], yn[k]);
                err[k] = fma(he, K[j][k], err[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < D; ++k) scatter(unew, D, k, yn[k]);
        scatter(unew, 1, ntraj * D, yn[D]);
        if (kfsal_out != nullptr) {
#pragma unroll
            for (int k = 0; k < D; ++k) scatter(kfsal_out, D, k, K[S - 1][k]);
            scatter(kfsal_out, 1, ntraj * D, K[S - 1][D]);
        }
        if (sumsq != nullptr) {
#pragma unroll
            for (int k = 0; k < N; ++k) {
                const V xs = yn[k] + err[k];
#pragma unroll
                for (int x = 0; x < W; ++x) {
                    if (!st[x]) continue;
                    const double un = (double)P::get(yn[k], x), xv = (double)P::get(xs, x);
                    const double tol = atol + rtol * fmax(fabs(un), fabs(xv));
                    const double rr = (un - xv) / tol;
                    local = fma(rr, rr, local);
                }
            }
        }
    }
    if (sumsq == nullptr) return;
    __shared__ double wsum[CNF_THREADS / 32];
    __shared__ bool is_last;
    local = warp_sum(local);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int wi = 0; wi < CNF_THREADS / 32; ++wi) s += wsum[wi];
        work->partial[blockIdx.x] = s;
        __threadfence();
        is_last = (atomicAdd(&work->ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __shared__ double sred[2];
        if (threadIdx.x < 32) {
            __threadfence();
            double s = 0.0;
            for (int b = threadIdx.x; b < (int)gridDim.x; b += 32) s += ((volatile double *)work->partial)[b];
            s = warp_sum(s);
            if (threadIdx.x == 0) sred[0] = s;
        }
        __syncthreads();
        if (dctl != nullptr && pc.peer_bufs != nullptr && pc.world > 1) {
            // sharded run: the verdict needs the error norm of the whole batch -- summed over the ranks here, through the
            // peers' inboxes (identical bits on every rank: they all take the same decision)
            PeerComm q = pc;
            q.epoch = dctl->epoch_next;
            peer_allreduce_and_store<double>(&sred[0], 1, q, &sred[1]);
            __syncthreads();
            if (threadIdx.x == 0) sred[0] = sred[1], dctl->epoch_next = q.epoch + 1ull;
        }
        if (threadIdx.x == 0) {
            const double s = sred[0];
            *sumsq = s;
            work->ticket = 0u;
            if (dctl != nullptr) {
                ctl::report(*dctl, s);
                __threadfence();
                if (loop_cond != 0ull) cudaGraphSetConditional(loop_cond, dctl->done == 0 ? 1u : 0u);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// adjoint sweep

constexpr int CNF_ADJ_WARPS = 4;
constexpr int CNF_ADJ_THREADS = CNF_ADJ_WARPS * 32;

// Shape of the warp-private reduction tile.  A warp carries NT = 32 W trajectories (W = Pack<T>::W per thread).  Phase 2
// turns the tile: lane = (hidden unit u, trajectory group g), HALVES = W groups of 32/W lanes, each lane summing the
// 16-byte vectors v = HALVES m + g of its unit's row -- so with two trajectories per thread the chunk holds 15 units and
// all but two lanes work, instead of 15 of 32.
template <typename T, int D, int H, int LPT>
struct CnfAdjShape {
    static constexpr int W = Pack<T>::W;
    static constexpr int NT = 32 * W / LPT;
    static constexpr int HALVES = W;
    static constexpr int LPH = 32 / HALVES;                      // lanes per trajectory group
    static constexpr int NCH = (W == 1) ? 2 : 4;                  // chunks of hidden units per stage
    static constexpr int JH = (H + NCH - 1) / NCH;                // 30 (fp64) / 15 (fp32) units per chunk
    static constexpr int VEC = 16 / sizeof(T);
    static constexpr int PITCH = NT + VEC;                        // 16-byte row skew: conflict-free vector loads in phase 2
    static constexpr int NP = 2 * H * D + 4 * H + 4 * D;
    static_assert(JH <= LPH, "chunk too wide");
};

struct CnfAdjWork {
    unsigned int ticket;
    unsigned int pad[15];
    double partial[1];  // [blocks][NP]
};

// warp-private tile: four per-(unit, trajectory) arrays + the per-trajectory vectors phase 2 needs.  (theta_j = dL/dg1_j =
// delta_j p_j + beta'_j q_j needs no array of its own: p_j = W1[j,:] z + b1_j and q_j = W1[j,:] e, so its sum over the
// trajectories is W1[j,:] . (sum delta_j z + sum beta'_j e) + b1_j sum delta_j -- quantities phase 2 forms anyway.)
template <typename T, int D, int H, int LPT>
struct alignas(16) CnfTile {
    T dl[CnfAdjShape<T, D, H, LPT>::JH * CnfAdjShape<T, D, H, LPT>::PITCH];  // delta_j  = dL/da_j
    T bp[CnfAdjShape<T, D, H, LPT>::JH * CnfAdjShape<T, D, H, LPT>::PITCH];  // beta'_j  = -v_l sg_j w_j
    T sp[CnfAdjShape<T, D, H, LPT>::JH * CnfAdjShape<T, D, H, LPT>::PITCH];  // s_j      = softplus(a_j)
    T eg[CnfAdjShape<T, D, H, LPT>::JH * CnfAdjShape<T, D, H, LPT>::PITCH];  // -v_l sg_j q_j g1_j
    T Z[D][CnfAdjShape<T, D, H, LPT>::NT], E[D][CnfAdjShape<T, D, H, LPT>::NT], VZ[D][CnfAdjShape<T, D, H, LPT>::NT];
};

template <typename T>
struct CnfVec;
template <>
struct CnfVec<float> {
    typedef float4 type;
};
template <>
struct CnfVec<double> {
    typedef double2 type;
};
template <typename T>
__device__ __forceinline__ void cnf_lds16(const T *p, T (&r)[16 / sizeof(T)]) {
    typename CnfVec<T>::type v = *reinterpret_cast<const typename CnfVec<T>::type *>(p);
    memcpy(r, &v, 16);
}

// the thread's W trajectories side by side in a tile row (column = W lane + x)
__device__ __forceinline__ void tile_put(double *row, int lane, double v) { row[lane] = v; }
__device__ __forceinline__ void tile_put(float *row, int lane, F2 v) {
    *reinterpret_cast<unsigned long long *>(row + 2 * lane) = v.v;
}
__device__ __forceinline__ double one_minus(double x) { return 1.0 - x; }
__device__ __forceinline__ F2 one_minus(F2 x) { return fma(x, -1.0f, 1.0f); }

// phase-2 accumulators: sums over a 16-byte vector of trajectories (fp32: the two halves of a packed register hold the
// partial sums of even / odd trajectories)
template <typename T>
struct VecAcc;
template <>
struct VecAcc<double> {
    typedef double A;
    static __device__ __forceinline__ A zero() { return 0.0; }
    static __device__ __forceinline__ void mac(A &acc, const double (&x)[2], const double (&y)[2]) {
        acc = fma(x[0], y[0], acc);
        acc = fma(x[1], y[1], acc);
    }
    static __device__ __forceinline__ void add(A &acc, const double (&x)[2]) { acc += x[0] + x[1]; }
    static __device__ __forceinline__ double total(A a) { return a; }
};
template <>
struct VecAcc<float> {
    typedef F2 A;
    static __device__ __forceinline__ A zero() { return splat(0.0f); }
    static __device__ __forceinline__ void mac(A &acc, const float (&x)[4], const float (&y)[4]) {
        acc = fma(pk(x[0], x[1]), pk(y[0], y[1]), acc);
        acc = fma(pk(x[2], x[3]), pk(y[2], y[3]), acc);
    }
    static __device__ __forceinline__ void add(A &acc, const float (&x)[4]) {
        acc = acc + pk(x[0], x[1]);
        acc = acc + pk(x[2], x[3]);
    }
    static __device__ __forceinline__ float total(A a) { return lo(a) + hi(a); }
};

template <typename T>
struct AccType {
    typedef double type;
};
template <>
struct AccType<float> {
    typedef float type;
};

template <typename T, int D, int H, int S, int LPT>
__global__ void __launch_bounds__(CNF_ADJ_THREADS)
cnf_rk_adj_kernel(const CnfPtrs<T> w, const pnode_rk_tableau tab, const int64_t ntraj,
                  const pnode_step *__restrict__ sched, const int nsteps_arg, const int last_slot,
                  const T *__restrict__ gout, const T *__restrict__ ckpt, T *__restrict__ lambda_out,
                  T *__restrict__ mu_out, CnfAdjWork *__restrict__ work, const PeerComm pc,
                  const int *__restrict__ d_nsteps) {
    const int nsteps = d_nsteps != nullptr ? *d_nsteps : nsteps_arg;  // device-resident schedule: the step count too
    typedef CnfAdjShape<T, D, H, LPT> Sh;
    typedef Pack<T> P;
    typedef typename P::V V;
    typedef VecAcc<T> VA;
    constexpr int JH = Sh::JH, PITCH = Sh::PITCH, NP = Sh::NP, VEC = Sh::VEC, NCH = Sh::NCH, W = Sh::W, NT = Sh::NT;
    constexpr int HALVES = Sh::HALVES, LPH = Sh::LPH;
    constexpr int NST = D + 1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CnfShared<T, D, H, S> &sm = *reinterpret_cast<CnfShared<T, D, H, S> *>(smem_raw);
    CnfTile<T, D, H, LPT> *tiles =
        reinterpret_cast<CnfTile<T, D, H, LPT> *>(smem_raw + ((sizeof(CnfShared<T, D, H, S>) + 15) / 16) * 16);
    __shared__ bool is_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int pu = lane % LPH, pg = lane / LPH;  // phase 2: hidden unit within the chunk, trajectory group
    CnfTile<T, D, H, LPT> &tile = tiles[warp];
    const int sub = lane % LPT, col = lane / LPT;  // share of the hidden units; the slot's column pair in the tile
    const int s_eff = tab.fsal ? S - 1 : S;
    const int64_t state_n = ntraj * NST;

    // per-lane accumulators, lane = (hidden unit of chunk c, trajectory group): [0,D) dW1 row, [D,2D) dW2 column, then
    // db1, dhb1, dhgw1, dhgb1.  They live in local memory (indexed by the chunk), are read into registers BEFORE the phase-2
    // loop and written back after it, so the L2 round trip hides behind the loop.  fp32 path: fp32 sums (each term is
    // already an fp32 sum over 32 trajectories; ~250 terms per lane and launch), converted for the fp64 block combine.
    typedef typename AccType<T>::type AccT;
    constexpr int NA = 2 * D + 4;
    AccT acc[NCH][NA];
#pragma unroll 1
    for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int x = 0; x < NA; ++x) acc[c][x] = AccT(0);
    // per-thread accumulators of the layer-2 bias / gate gradients (reduced over the warp at the end)
    T aB2[D], aHB2[D], aHGW2[D], aHGB2[D];
#pragma unroll
    for (int k = 0; k < D; ++k) aB2[k] = aHB2[k] = aHGW2[k] = aHGB2[k] = T(0);
    auto both_lanes = [](V v) -> T {
        T t = P::get(v, 0);
        if (W == 2) t += P::get(v, 1);
        return t;
    };

    const int64_t nslots = (ntraj + W - 1) / W;
    constexpr int SLOTS_PER_CTA = CNF_ADJ_THREADS / LPT;
    const int64_t ntiles = (nslots + SLOTS_PER_CTA - 1) / SLOTS_PER_CTA;
    for (int64_t tidx = blockIdx.x; tidx < ntiles; tidx += gridDim.x) {
        const int64_t slot = tidx * SLOTS_PER_CTA + threadIdx.x / LPT;
        // the thread's trajectories; the ones past the end carry zeros everywhere, which contribute nothing to any sum
        int64_t tr[W];
        bool ok[W];
#pragma unroll
        for (int x = 0; x < W; ++x) {
            tr[x] = slot * W + x;
            ok[x] = tr[x] < ntraj;
            if (!ok[x]) tr[x] = 0;
        }
        auto gather = [&](const T *base, int64_t mul, int64_t off) -> V {
            T v[2] = {T(0), T(0)};
#pragma unroll
            for (int x = 0; x < W; ++x) v[x] = ok[x] ? base[tr[x] * mul + off] : T(0);
            return P::make(v[0], v[1]);
        };
        V lam[NST], e[D];
#pragma unroll
        for (int k = 0; k < D; ++k) {
            lam[k] = gather(gout, D, (int64_t)last_slot * state_n + k);
            e[k] = gather(w.e, D, k);
        }
        lam[D] = gather(gout, 1, (int64_t)last_slot * state_n + ntraj * D);
        // stage checkpoints are fetched one stage ahead of their use
        const int i_first = tab.fsal ? S - 2 : S - 1;
        V znext[D];
#pragma unroll
        for (int k = 0; k < D; ++k)
            znext[k] = gather(ckpt, 1, (((int64_t)(nsteps - 1) * s_eff + i_first) * D + k) * ntraj);

        for (int n = nsteps - 1; n >= 0; --n) {
            const double h = sched[n].h;
            const double t = sched[n].t;
            const int in_slot = sched[n].in_slot;
            __syncthreads();  // every warp is done with the previous step's gates
            cnf_setup<T, D, H, S>(sm, w, tab, t, h);
            __syncthreads();
            V ls[S][D];
#pragma unroll 1
            for (int i = S - 1; i >= 0; --i) {
                if (tab.fsal && i == S - 1) {
#pragma unroll
                    for (int k = 0; k < D; ++k) ls[i][k] = P::all(T(0));
                    continue;
                }
                // cotangents of the stage slope (SURVEY.md A.4), pre-multiplied by the step coefficient
                const bool has_b = sm.adj_has_b[i] != 0;
                const T cstep = sm.adj_c[i];
                V vz[D];
#pragma unroll
                for (int k = 0; k < D; ++k) vz[k] = has_b ? lam[k] : P::all(T(0));
                for (int j = i + 1; j < S; ++j) {
                    const T rr = sm.adj_r[j][i];
#pragma unroll
                    for (int k = 0; k < D; ++k) vz[k] = fma(rr, ls[j][k], vz[k]);
                }
                // the logp row of the Jacobian is zero: its stage adjoints vanish, only lambda_logp itself feeds v_l
                const V mvl = has_b ? lam[D] * (-cstep) : P::all(T(0));  // = -v_l
                V z[D], vg[D], ge[D], r[D], rho[D], dzk[D];
                const T tt = sm.tstage[i];
#pragma unroll
                for (int k = 0; k < D; ++k) z[k] = znext[k];
                const int nn = i > 0 ? n : n - 1, in = i > 0 ? i - 1 : i_first;
                if (nn >= 0) {
#pragma unroll
                    for (int k = 0; k < D; ++k) znext[k] = gather(ckpt, 1, (((int64_t)nn * s_eff + in) * D + k) * ntraj);
                }
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    vz[k] = vz[k] * cstep;
                    vg[k] = vz[k] * sm.g2[i][k];
                    ge[k] = sm.g2[i][k] * e[k];
                    rho[k] = P::all(T(0));
                    dzk[k] = P::all(T(0));
                    r[k] = P::all(sub == 0 ? sm.b2[k] : T(0));
                    if (sub == 0) {
                        tile_put(tile.Z[k], col, z[k]);
                        tile_put(tile.E[k], col, e[k]);
                        tile_put(tile.VZ[k], col, vz[k]);
                    }
                }
#pragma unroll 1
                for (int c = 0; c < NCH; ++c) {
                    const int j0 = c * JH;
                    const int jn = (H - j0 < JH) ? (H - j0) : JH;
                    // ---- phase 1 (lane = W trajectories) --------------------------------------------------------------
                    CNF_UNROLL(CNF_P1_UNROLL)
                    for (int jj = sub; jj < jn; jj += LPT) {
                        const int j = j0 + jj;
                        const UnitC<T, D> u = sm.unit[j];
                        V p = P::all(u.b1), q = P::all(T(0)), ww = P::all(T(0)), m = P::all(T(0));
#pragma unroll
                        for (int k = 0; k < D; ++k) {
                            p = fma(u.w1[k], z[k], p);
                            q = fma(u.w1[k], e[k], q);
                            ww = fma(u.w2[k], ge[k], ww);
                            m = fma(u.w2[k], vg[k], m);
                        }
                        const T g1 = sm.g1[i][j];
                        const V a = fma(p, g1, sm.c1[i][j]);
                        V s, sg;
                        softplus_sigmoid(a, s, sg);
#pragma unroll
                        for (int k = 0; k < D; ++k) r[k] = fma(u.w2[k], s, r[k]);
                        const V bq = mvl * sg;     // -v_l sg
                        const V betap = bq * ww;   // d(-v_l div)/d(g1 q) per unit
                        const V epsp = bq * q;
                        const V delta = fma(betap * g1 * q, one_minus(sg), m * sg);  // dL/da_j
                        const V dg = delta * g1;
                        const V egv = epsp * g1;
#pragma unroll
                        for (int k = 0; k < D; ++k) {
                            dzk[k] = fma(u.w1[k], dg, dzk[k]);
                            rho[k] = fma(u.w2[k], egv, rho[k]);
                        }
                        tile_put(&tile.dl[jj * PITCH], col, delta);
                        tile_put(&tile.bp[jj * PITCH], col, betap);
                        tile_put(&tile.sp[jj * PITCH], col, s);
                        tile_put(&tile.eg[jj * PITCH], col, egv);
                    }
                    __syncwarp();
                    // ---- phase 2 (lane = hidden unit x trajectory group): sums over the warp's trajectories -----------
                    if (pu < jn) {
                        // the chunk's accumulators are read before the loop (fp32) so that their load hides behind it;
                        // fp64 has no registers to spare for that and reads them after the loop
                        constexpr bool EARLY = W == 2;
                        AccT ar[NA];
                        if (EARLY) {
#pragma unroll
                            for (int x = 0; x < NA; ++x) ar[x] = acc[c][x];
                        }
                        typename VA::A sW1[D], sW2[D], sD = VA::zero();
#pragma unroll
                        for (int k = 0; k < D; ++k) sW1[k] = sW2[k] = VA::zero();
                        CNF_UNROLL(CNF_P2_UNROLL)
                        for (int mm = 0; mm < NT / VEC / HALVES; ++mm) {
                            const int kk = (mm * HALVES + pg) * VEC;
                            T dl[VEC], bp[VEC], sp[VEC], eg[VEC];
                            cnf_lds16(&tile.dl[pu * PITCH + kk], dl);
                            cnf_lds16(&tile.bp[pu * PITCH + kk], bp);
                            cnf_lds16(&tile.sp[pu * PITCH + kk], sp);
                            cnf_lds16(&tile.eg[pu * PITCH + kk], eg);
                            VA::add(sD, dl);
#pragma unroll
                            for (int k = 0; k < D; ++k) {
                                T zz[VEC], ee[VEC], vv[VEC];
                                cnf_lds16(&tile.Z[k][kk], zz);
                                cnf_lds16(&tile.E[k][kk], ee);
                                cnf_lds16(&tile.VZ[k][kk], vv);
                                VA::mac(sW1[k], dl, zz);
                                VA::mac(sW1[k], bp, ee);
                                VA::mac(sW2[k], vv, sp);
                                VA::mac(sW2[k], eg, ee);
                            }
                        }
                        if (!EARLY) {
#pragma unroll
                            for (int x = 0; x < NA; ++x) ar[x] = acc[c][x];
                        }
                        const AccT g1 = (AccT)sm.g1[i][j0 + pu];
                        const AccT gd = g1 * (AccT(1) - g1);
                        const AccT dD = (AccT)VA::total(sD), ta = (AccT)tt;
                        const UnitC<T, D> un = sm.unit[j0 + pu];
                        AccT dTh = (AccT)un.b1 * dD;  // sum over the trajectories of theta_j
#pragma unroll
                        for (int k = 0; k < D; ++k) {
                            const AccT s1 = (AccT)VA::total(sW1[k]);
                            dTh = fma((AccT)un.w1[k], s1, dTh);
                            ar[k] = fma(g1, s1, ar[k]);
                            ar[D + k] = fma((AccT)sm.g2[i][k], (AccT)VA::total(sW2[k]), ar[D + k]);
                        }
                        ar[2 * D] = fma(g1, dD, ar[2 * D]);
                        ar[2 * D + 1] = fma(ta, dD, ar[2 * D + 1]);
                        ar[2 * D + 2] = fma(ta * gd, dTh, ar[2 * D + 2]);
                        ar[2 * D + 3] = fma(gd, dTh, ar[2 * D + 3]);
#pragma unroll
                        for (int x = 0; x < NA; ++x) acc[c][x] = ar[x];
                    }
                    __syncwarp();
                }
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    dzk[k] = sub_sum<LPT>(dzk[k]);
                    r[k] = sub_sum<LPT>(r[k]);
                    rho[k] = sub_sum<LPT>(rho[k]);
                    ls[i][k] = dzk[k];
                    const T g2 = sm.g2[i][k];
                    const V Gk = fma(vz[k], r[k], e[k] * rho[k]) * (g2 * (T(1) - g2));  // dL/d(gate-2 pre-activation)
                    if (sub != 0) continue;  // one lane of the slot feeds the per-thread sums
                    const T svg = both_lanes(vg[k]), svz = both_lanes(vz[k]), sG = both_lanes(Gk);
                    aB2[k] += svg;
                    aHB2[k] = fma(svz, tt, aHB2[k]);
                    aHGB2[k] += sG;
                    aHGW2[k] = fma(sG, tt, aHGW2[k]);
                }
            }
            for (int i = 0; i < S; ++i)
#pragma unroll
                for (int k = 0; k < D; ++k) lam[k] += ls[i][k];
            if (in_slot >= 0) {
#pragma unroll
                for (int k = 0; k < D; ++k) lam[k] += gather(gout, D, (int64_t)in_slot * state_n + k);
                lam[D] += gather(gout, 1, (int64_t)in_slot * state_n + ntraj * D);
            }
        }
#pragma unroll
        for (int x = 0; x < W; ++x) {
            if (!ok[x] || sub != 0) continue;
#pragma unroll
            for (int k = 0; k < D; ++k) lambda_out[tr[x] * D + k] = P::get(lam[k], x);
            lambda_out[ntraj * D + tr[x]] = P::get(lam[D], x);
        }
    }

    // ---- combine: per-lane / per-thread accumulators -> block partial (fixed order) -> last block sums the grid ---------
    __syncthreads();
    double *blk = reinterpret_cast<double *>(tiles);  // [CNF_ADJ_WARPS][NP]
    // (the launcher sizes the dynamic shared memory for whichever is larger: the tiles or this combine buffer)
    constexpr int O_B1 = H * D, O_HB1 = O_B1 + H, O_HGW1 = O_HB1 + H, O_HGB1 = O_HGW1 + H, O_W2 = O_HGB1 + H,
                  O_B2 = O_W2 + D * H, O_HB2 = O_B2 + D, O_HGW2 = O_HB2 + D, O_HGB2 = O_HGW2 + D;
    // the trajectory groups of a unit sit LPH lanes apart: group 0 collects
    auto both = [&](double v) -> double {
        if (HALVES == 2) v += __shfl_down_sync(0xffffffffu, v, LPH);
        return v;
    };
    for (int c = 0; c < NCH; ++c) {
        const int j = c * JH + pu;
        const bool writer = pg == 0 && pu < JH && j < H;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const double v1 = both((double)acc[c][k]), v2 = both((double)acc[c][D + k]);
            if (writer) {
                blk[warp * NP + j * D + k] = v1;
                blk[warp * NP + O_W2 + k * H + j] = v2;
            }
        }
        const double b1 = both((double)acc[c][2 * D]), hb1 = both((double)acc[c][2 * D + 1]);
        const double hgw1 = both((double)acc[c][2 * D + 2]), hgb1 = both((double)acc[c][2 * D + 3]);
        if (writer) {
            blk[warp * NP + O_B1 + j] = b1;
            blk[warp * NP + O_HB1 + j] = hb1;
            blk[warp * NP + O_HGW1 + j] = hgw1;
            blk[warp * NP + O_HGB1 + j] = hgb1;
        }
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const double b2 = warp_sum((double)aB2[k]), hb2 = warp_sum((double)aHB2[k]);
        const double hgw2 = warp_sum((double)aHGW2[k]), hgb2 = warp_sum((double)aHGB2[k]);
        if (lane == 0) {
            blk[warp * NP + O_B2 + k] = b2;
            blk[warp * NP + O_HB2 + k] = hb2;
            blk[warp * NP + O_HGW2 + k] = hgw2;
            blk[warp * NP + O_HGB2 + k] = hgb2;
        }
    }
    __syncthreads();
    for (int p = threadIdx.x; p < NP; p += blockDim.x) {
        double s = 0.0;
#pragma unroll
        for (int wi = 0; wi < CNF_ADJ_WARPS; ++wi) s += blk[wi * NP + p];
        work->partial[(int64_t)blockIdx.x * NP + p] = s;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(&work->ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (is_last) {
        __threadfence();
        const bool dp = pc.peer_bufs != nullptr && pc.world > 1;
        for (int p = threadIdx.x; p < NP; p += blockDim.x) {
            double s = 0.0;
            for (int b = 0; b < (int)gridDim.x; ++b) s += ((volatile double *)work->partial)[(int64_t)b * NP + p];
            if (dp)
                blk[p] = s;
            else
                mu_out[p] = (T)s;
        }
        if (threadIdx.x == 0) work->ticket = 0u;
        if (dp) {
            __syncthreads();
            peer_allreduce_and_store<T>(blk, NP, pc, mu_out);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// host dispatch

// states at the output times of a solve that ran without the host: slot k < nout - 1 from the solution buffer (copied there
// by the attempt that followed the hit), the last one from the current state buffer; NaN if the attempt budget ran out
template <typename T>
__global__ void cnf_gather_kernel(const pnode_cnf_ctl *__restrict__ c, const T *__restrict__ ubuf, const T *__restrict__ sol,
                                  T *__restrict__ out, int nout, int64_t n) {
    const int k = nout == 1 ? 0 : 1 + (int)blockIdx.y;  // nout == 1: single end time, out[0] is the final state
    const bool last = k == nout - 1;
    const bool finished = c->done == 1;
    const T *src = last ? ubuf + (int64_t)c->cur * n : sol + (int64_t)k * n;
    const T bad = (T)NAN;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[(int64_t)k * n + i] = finished ? src[i] : bad;
}

__global__ void ctl_probe_kernel(pnode_cnf_ctl *c, const double *sumsq, int n) {
    for (int i = 0; i < n && c->done == 0; ++i) ctl::report(*c, sumsq[i]);
}

static bool cnf_shape_ok(int dim, int hidden, int stages) {
    return dim == 6 && hidden == 60 && (stages == 4 || stages == 7 || stages == 1 || stages == 2 || stages == 3);
}

template <typename T>
static CnfPtrs<T> cnf_ptrs(const pnode_cnf_desc *c) {
    auto p = [](const void *x) { return static_cast<const T *>(x); };
    return CnfPtrs<T>{p(c->d_w1), p(c->d_b1), p(c->d_hb1), p(c->d_hgw1), p(c->d_hgb1), p(c->d_w2),
                      p(c->d_b2), p(c->d_hb2), p(c->d_hgw2), p(c->d_hgb2), p(c->d_e), c->t_via_f32};
}

// Small batches spread a trajectory slot over CNF_SMALL_LPT lanes: below this many slots the GPU has idle lanes to spare
// and the launch is bound by the dependent chain of one thread, not by throughput.
constexpr int CNF_SMALL_LPT = 4;
template <typename T>
static bool cnf_small_batch(int64_t ntraj) {
    const int64_t nslots = (ntraj + Pack<T>::W - 1) / Pack<T>::W;
    return nslots * CNF_SMALL_LPT <= (int64_t)sm_count() * 256;
}

template <typename T, int S, int LPT>
static int launch_cnf_attempt_lpt(const pnode_cnf_desc *c, const pnode_rk_tableau *tab, const void *d_u, const void *d_kin,
                                  int64_t ntraj, double t, double h, void *d_unew, void *d_kout, void *d_ckpt, double atol,
                                  double rtol, double *d_sumsq, void *d_work, cudaStream_t st, pnode_cnf_ctl *d_ctl,
                                  void *d_ubuf, void *d_kbuf, int64_t ckpt_step_elems, void *d_sol, int nlaunch,
                                  unsigned long long loop_cond, const PeerComm &pc) {
    auto kern = cnf_rk_attempt_kernel<T, 6, 60, S, LPT>;
    const size_t smem = sizeof(typename Pack<T>::V) * 60 * CNF_THREADS;  // q_j columns
    static int ctas_per_sm = 0;
    if (ctas_per_sm == 0) {
        PNODE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        PNODE_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kern, CNF_THREADS, smem));
        if (ctas_per_sm < 1) ctas_per_sm = 1;
    }
    const int64_t nslots = (ntraj + Pack<T>::W - 1) / Pack<T>::W;  // fp32: two trajectories per thread (csrc/f32x2.cuh)
    int64_t want = (nslots * LPT + CNF_THREADS - 1) / CNF_THREADS;
    int64_t cap = (int64_t)sm_count() * ctas_per_sm;
    if (cap > CNF_MAX_BLOCKS) cap = CNF_MAX_BLOCKS;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    for (int l = 0; l < nlaunch; ++l)
        kern<<<grid, CNF_THREADS, smem, st>>>(cnf_ptrs<T>(c), *tab, static_cast<const T *>(d_u), static_cast<const T *>(d_kin),
                                           ntraj, t, h, static_cast<T *>(d_unew), static_cast<T *>(d_kout),
                                           static_cast<T *>(d_ckpt), atol, rtol, d_sumsq,
                                           static_cast<CnfWrmsWork *>(d_work), d_ctl, static_cast<T *>(d_ubuf),
                                           static_cast<T *>(d_kbuf), ckpt_step_elems, static_cast<T *>(d_sol), loop_cond, pc);
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

template <typename T, int S>
static int launch_cnf_attempt(const pnode_cnf_desc *c, const pnode_rk_tableau *tab, const void *d_u, const void *d_kin,
                              int64_t ntraj, double t, double h, void *d_unew, void *d_kout, void *d_ckpt, double atol,
                              double rtol, double *d_sumsq, void *d_work, cudaStream_t st, pnode_cnf_ctl *d_ctl = nullptr,
                              void *d_ubuf = nullptr, void *d_kbuf = nullptr, int64_t ckpt_step_elems = 0,
                              void *d_sol = nullptr, int nlaunch = 1, unsigned long long loop_cond = 0ull,
                              const PeerComm &pc = PeerComm{nullptr, 0, 1, 0ull}) {
    if (cnf_small_batch<T>(ntraj))
        return launch_cnf_attempt_lpt<T, S, CNF_SMALL_LPT>(c, tab, d_u, d_kin, ntraj, t, h, d_unew, d_kout, d_ckpt, atol, rtol,
                                                           d_sumsq, d_work, st, d_ctl, d_ubuf, d_kbuf, ckpt_step_elems,
                                                           d_sol, nlaunch, loop_cond, pc);
    return launch_cnf_attempt_lpt<T, S, 1>(c, tab, d_u, d_kin, ntraj, t, h, d_unew, d_kout, d_ckpt, atol, rtol, d_sumsq,
                                           d_work, st, d_ctl, d_ubuf, d_kbuf, ckpt_step_elems, d_sol, nlaunch, loop_cond, pc);
}

template <typename T, int S, int LPT>
static int launch_cnf_adjoint_lpt(const pnode_cnf_desc *c, const pnode_rk_tableau *tab, int64_t ntraj,
                                  const pnode_step *d_sched, int nsteps, int last_slot, const void *d_gout,
                                  const void *d_ckpt, void *d_lambda, void *d_mu, void *d_work, const PeerComm &pc,
                                  cudaStream_t st, const int *d_nsteps) {
    auto kern = cnf_rk_adj_kernel<T, 6, 60, S, LPT>;
    constexpr size_t tiles = sizeof(CnfTile<T, 6, 60, LPT>) * CNF_ADJ_WARPS;
    constexpr size_t comb = sizeof(double) * CNF_ADJ_WARPS * CnfAdjShape<T, 6, 60, LPT>::NP;  // block combine reuses the tiles
    const size_t smem = ((sizeof(CnfShared<T, 6, 60, S>) + 15) / 16) * 16 + (tiles > comb ? tiles : comb);
    static int ctas_per_sm = 0;
    if (ctas_per_sm == 0) {
        PNODE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        PNODE_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kern, CNF_ADJ_THREADS, smem));
        if (ctas_per_sm < 1) ctas_per_sm = 1;
    }
    const int64_t nslots = (ntraj + Pack<T>::W - 1) / Pack<T>::W;
    int64_t want = (nslots * LPT + CNF_ADJ_THREADS - 1) / CNF_ADJ_THREADS;
    int64_t cap = (int64_t)sm_count() * ctas_per_sm;
    if (cap > CNF_MAX_BLOCKS) cap = CNF_MAX_BLOCKS;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, CNF_ADJ_THREADS, smem, st>>>(cnf_ptrs<T>(c), *tab, ntraj, d_sched, nsteps, last_slot,
                                              static_cast<const T *>(d_gout), static_cast<const T *>(d_ckpt),
                                              static_cast<T *>(d_lambda), static_cast<T *>(d_mu),
                                              static_cast<CnfAdjWork *>(d_work), pc, d_nsteps);
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

template <typename T, int S>
static int launch_cnf_adjoint(const pnode_cnf_desc *c, const pnode_rk_tableau *tab, int64_t ntraj,
                              const pnode_step *d_sched, int nsteps, int last_slot, const void *d_gout,
                              const void *d_ckpt, void *d_lambda, void *d_mu, void *d_work, const PeerComm &pc,
                              cudaStream_t st, const int *d_nsteps = nullptr) {
    if (cnf_small_batch<T>(ntraj))
        return launch_cnf_adjoint_lpt<T, S, CNF_SMALL_LPT>(c, tab, ntraj, d_sched, nsteps, last_slot, d_gout, d_ckpt,
                                                           d_lambda, d_mu, d_work, pc, st, d_nsteps);
    return launch_cnf_adjoint_lpt<T, S, 1>(c, tab, ntraj, d_sched, nsteps, last_slot, d_gout, d_ckpt, d_lambda, d_mu, d_work,
                                           pc, st, d_nsteps);
}

}  // namespace pnode

using namespace pnode;

#define PNODE_CNF_STAGES(X) X(1) X(2) X(3) X(4) X(7)

extern "C" {

int pnode_cnf_rk_supported(int dim, int hidden, int dtype, int stages) {
    return (dtype == PNODE_F32 || dtype == PNODE_F64) && cnf_shape_ok(dim, hidden, stages) ? 1 : 0;
}

int pnode_cnf_rk_attempt(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, const void *d_u,
                         const void *d_kfsal_in, int64_t ntraj, double t, double h, void *d_unew, void *d_kfsal_out,
                         void *d_ckpt, double atol, double rtol, double *d_sumsq, void *d_work, void *stream) {
    PNODE_REQUIRE(cnf && tab && d_u && d_unew, "pnode_cnf_rk_attempt: null argument");
    PNODE_REQUIRE(cnf_shape_ok(cnf->dim, cnf->hidden, tab->s), "pnode_cnf_rk_attempt: unsupported shape D=%d H=%d s=%d",
                  cnf->dim, cnf->hidden, tab->s);
    PNODE_REQUIRE(d_sumsq == nullptr || (tab->has_be && d_work != nullptr),
                  "pnode_cnf_rk_attempt: error norm needs an embedded tableau and a work buffer");
    if (ntraj == 0) {
        if (d_sumsq) PNODE_CUDA_OK(cudaMemsetAsync(d_sumsq, 0, sizeof(double), static_cast<cudaStream_t>(stream)));
        return 0;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
#define X(SS)                                                                                                       \
    if (tab->s == SS) {                                                                                             \
        if (cnf->dtype == PNODE_F32)                                                                                \
            return launch_cnf_attempt<float, SS>(cnf, tab, d_u, d_kfsal_in, ntraj, t, h, d_unew, d_kfsal_out, d_ckpt, \
                                                 atol, rtol, d_sumsq, d_work, st);                                  \
        return launch_cnf_attempt<double, SS>(cnf, tab, d_u, d_kfsal_in, ntraj, t, h, d_unew, d_kfsal_out, d_ckpt,   \
                                              atol, rtol, d_sumsq, d_work, st);                                     \
    }
    PNODE_CNF_STAGES(X)
#undef X
    PNODE_REQUIRE(false, "pnode_cnf_rk_attempt: no kernel for %d stages", tab->s);
}

int pnode_cnf_rk_attempts_ctl(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, void *d_ubuf, void *d_kbuf,
                              int64_t ntraj, void *d_ckpt_base, int64_t ckpt_step_elems, void *d_sol, double atol,
                              double rtol, pnode_cnf_ctl *d_ctl, void *d_work, int nlaunch, void *stream) {
    PNODE_REQUIRE(cnf && tab && d_ubuf && d_ctl && d_work, "pnode_cnf_rk_attempts_ctl: null argument");
    PNODE_REQUIRE(cnf_shape_ok(cnf->dim, cnf->hidden, tab->s), "pnode_cnf_rk_attempts_ctl: unsupported shape D=%d H=%d s=%d",
                  cnf->dim, cnf->hidden, tab->s);
    PNODE_REQUIRE(tab->has_be, "pnode_cnf_rk_attempts_ctl: the device controller needs an embedded tableau");
    PNODE_REQUIRE(!tab->fsal || d_kbuf, "pnode_cnf_rk_attempts_ctl: FSAL tableau without slope buffers");
    PNODE_REQUIRE(ntraj > 0 && nlaunch >= 1 && nlaunch <= 64, "pnode_cnf_rk_attempts_ctl: bad ntraj / nlaunch");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    double *d_sumsq = &d_ctl->sumsq;  // consumed on the device by the controller
#define X(SS)                                                                                                         \
    if (tab->s == SS) {                                                                                               \
        if (cnf->dtype == PNODE_F32)                                                                                  \
            return launch_cnf_attempt<float, SS>(cnf, tab, nullptr, nullptr, ntraj, 0.0, 0.0, nullptr, nullptr, d_ckpt_base, \
                                                 atol, rtol, d_sumsq, d_work, st, d_ctl, d_ubuf, d_kbuf, ckpt_step_elems,    \
                                                 d_sol, nlaunch);                                                      \
        return launch_cnf_attempt<double, SS>(cnf, tab, nullptr, nullptr, ntraj, 0.0, 0.0, nullptr, nullptr, d_ckpt_base,    \
                                              atol, rtol, d_sumsq, d_work, st, d_ctl, d_ubuf, d_kbuf, ckpt_step_elems,       \
                                              d_sol, nlaunch);                                                         \
    }
    PNODE_CNF_STAGES(X)
#undef X
    PNODE_REQUIRE(false, "pnode_cnf_rk_attempts_ctl: no kernel for %d stages", tab->s);
}

// ---- the adaptive time loop as a CUDA graph with a device-driven WHILE node ---------------------------------------------
namespace {
struct CnfLoopKey {
    pnode_cnf_desc cnf;
    pnode_rk_tableau tab;
    void *ubuf, *kbuf, *ckpt, *sol, *ctl, *work;
    int64_t ntraj, ckpt_step_elems;
    double atol, rtol;
    const unsigned long long *peer_bufs;
    int rank, world;
};
struct CnfLoopGraph {
    CnfLoopKey key;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    unsigned long long last_use = 0;
};
constexpr int CNF_LOOP_CACHE = 8;
CnfLoopGraph g_loops[CNF_LOOP_CACHE];
unsigned long long g_loop_clock = 0;
cudaStream_t g_loop_capture_stream = nullptr;
std::mutex g_loop_mutex;

int build_loop_graph(const CnfLoopKey &k, CnfLoopGraph &out) {
    if (out.exec != nullptr) cudaGraphExecDestroy(out.exec);
    if (out.graph != nullptr) cudaGraphDestroy(out.graph);
    out.exec = nullptr, out.graph = nullptr;
    if (g_loop_capture_stream == nullptr)
        PNODE_CUDA_OK(cudaStreamCreateWithFlags(&g_loop_capture_stream, cudaStreamNonBlocking));
    PNODE_CUDA_OK(cudaGraphCreate(&out.graph, 0));
    cudaGraphConditionalHandle cond;
    PNODE_CUDA_OK(cudaGraphConditionalHandleCreate(&cond, out.graph, 1u, cudaGraphCondAssignDefault));
    cudaGraphNodeParams np = {};
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = cond;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    cudaGraphNode_t node;
    PNODE_CUDA_OK(cudaGraphAddNode(&node, out.graph, nullptr, 0, &np));
    cudaGraph_t body = np.conditional.phGraph_out[0];
    PNODE_CUDA_OK(cudaStreamBeginCaptureToGraph(g_loop_capture_stream, body, nullptr, nullptr, 0,
                                                cudaStreamCaptureModeRelaxed));
    int rc = -1;
    double *d_sumsq = &static_cast<pnode_cnf_ctl *>(k.ctl)->sumsq;
    const PeerComm pc{k.peer_bufs, k.rank, k.world, 0ull};  // the collective number lives in the control block
#define X(SS)                                                                                                            \
    if (k.tab.s == SS) {                                                                                                 \
        rc = k.cnf.dtype == PNODE_F32                                                                                    \
                 ? launch_cnf_attempt<float, SS>(&k.cnf, &k.tab, nullptr, nullptr, k.ntraj, 0.0, 0.0, nullptr, nullptr,  \
                                                 k.ckpt, k.atol, k.rtol, d_sumsq, k.work, g_loop_capture_stream,         \
                                                 static_cast<pnode_cnf_ctl *>(k.ctl), k.ubuf, k.kbuf, k.ckpt_step_elems, \
                                                 k.sol, 1, (unsigned long long)cond, pc)                                \
                 : launch_cnf_attempt<double, SS>(&k.cnf, &k.tab, nullptr, nullptr, k.ntraj, 0.0, 0.0, nullptr, nullptr, \
                                                  k.ckpt, k.atol, k.rtol, d_sumsq, k.work, g_loop_capture_stream,        \
                                                  static_cast<pnode_cnf_ctl *>(k.ctl), k.ubuf, k.kbuf,                   \
                                                  k.ckpt_step_elems, k.sol, 1, (unsigned long long)cond, pc);           \
    }
    PNODE_CNF_STAGES(X)
#undef X
    cudaError_t e = cudaStreamEndCapture(g_loop_capture_stream, nullptr);
    if (rc != 0) return rc;
    PNODE_CUDA_OK(e);
    PNODE_CUDA_OK(cudaGraphInstantiate(&out.exec, out.graph, 0));
    out.key = k;
    return 0;
}
}  // namespace

int pnode_cnf_rk_gather_ctl(const pnode_cnf_ctl *d_ctl, const void *d_ubuf, const void *d_sol, void *d_out, int nout,
                            int64_t n, int dtype, void *stream) {
    PNODE_REQUIRE(d_ctl && d_ubuf && d_out && nout >= 1 && n > 0, "pnode_cnf_rk_gather_ctl: bad argument");
    PNODE_REQUIRE(nout <= 2 || d_sol, "pnode_cnf_rk_gather_ctl: interior output times without the solution buffer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int grid = (int)((n + 255) / 256 < 1024 ? (n + 255) / 256 : 1024);
    if (dtype == PNODE_F32)
        cnf_gather_kernel<float><<<dim3(grid, nout - 1 > 0 ? nout - 1 : 1), 256, 0, st>>>(
            d_ctl, static_cast<const float *>(d_ubuf), static_cast<const float *>(d_sol), static_cast<float *>(d_out), nout, n);
    else if (dtype == PNODE_F64)
        cnf_gather_kernel<double><<<dim3(grid, nout - 1 > 0 ? nout - 1 : 1), 256, 0, st>>>(
            d_ctl, static_cast<const double *>(d_ubuf), static_cast<const double *>(d_sol), static_cast<double *>(d_out), nout,
            n);
    else
        PNODE_REQUIRE(false, "pnode_cnf_rk_gather_ctl: unsupported dtype %d", dtype);
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

int pnode_cnf_rk_adjoint_ctl(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, int64_t ntraj, const pnode_cnf_ctl *d_ctl,
                             int last_slot, const void *d_gout, const void *d_ckpt, void *d_lambda, void *d_mu, void *d_work,
                             void *stream) {
    PNODE_REQUIRE(cnf && tab && d_ctl && d_work && d_ckpt, "pnode_cnf_rk_adjoint_ctl: null argument");
    PNODE_REQUIRE(cnf_shape_ok(cnf->dim, cnf->hidden, tab->s), "pnode_cnf_rk_adjoint_ctl: unsupported shape D=%d H=%d s=%d",
                  cnf->dim, cnf->hidden, tab->s);
    const PeerComm pc{nullptr, 0, 1, 0ull};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
#define X(SS)                                                                                                            \
    if (tab->s == SS) {                                                                                                  \
        if (cnf->dtype == PNODE_F32)                                                                                     \
            return launch_cnf_adjoint<float, SS>(cnf, tab, ntraj, d_ctl->sched, 0, last_slot, d_gout, d_ckpt, d_lambda,  \
                                                 d_mu, d_work, pc, st, &d_ctl->steps);                                   \
        return launch_cnf_adjoint<double, SS>(cnf, tab, ntraj, d_ctl->sched, 0, last_slot, d_gout, d_ckpt, d_lambda,     \
                                              d_mu, d_work, pc, st, &d_ctl->steps);                                      \
    }
    PNODE_CNF_STAGES(X)
#undef X
    PNODE_REQUIRE(false, "pnode_cnf_rk_adjoint_ctl: no kernel for %d stages", tab->s);
}

int pnode_cnf_ctl_probe(pnode_cnf_ctl *d_ctl, const double *d_sumsq, int n, void *stream) {
    PNODE_REQUIRE(d_ctl && d_sumsq && n >= 0, "pnode_cnf_ctl_probe: bad argument");
    ctl_probe_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(d_ctl, d_sumsq, n);
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

int pnode_cnf_rk_solve_ctl(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, void *d_ubuf, void *d_kbuf,
                           int64_t ntraj, void *d_ckpt_base, int64_t ckpt_step_elems, void *d_sol, double atol, double rtol,
                           pnode_cnf_ctl *d_ctl, void *d_work, void *stream) {
    return pnode_cnf_rk_solve_ctl_dp(cnf, tab, d_ubuf, d_kbuf, ntraj, d_ckpt_base, ckpt_step_elems, d_sol, atol, rtol, d_ctl,
                                     d_work, nullptr, 0, 1, stream);
}

int pnode_cnf_rk_solve_ctl_dp(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, void *d_ubuf, void *d_kbuf,
                              int64_t ntraj, void *d_ckpt_base, int64_t ckpt_step_elems, void *d_sol, double atol, double rtol,
                              pnode_cnf_ctl *d_ctl, void *d_work, const uint64_t *d_peer_bufs, int rank, int world,
                              void *stream) {
    PNODE_REQUIRE(cnf && tab && d_ubuf && d_ctl && d_work, "pnode_cnf_rk_solve_ctl: null argument");
    PNODE_REQUIRE(world <= 1 || d_peer_bufs == nullptr || (rank >= 0 && rank < world && world <= 64),
                  "pnode_cnf_rk_solve_ctl_dp: bad rank/world");
    PNODE_REQUIRE(cnf_shape_ok(cnf->dim, cnf->hidden, tab->s), "pnode_cnf_rk_solve_ctl: unsupported shape D=%d H=%d s=%d",
                  cnf->dim, cnf->hidden, tab->s);
    PNODE_REQUIRE(tab->has_be, "pnode_cnf_rk_solve_ctl: the device controller needs an embedded tableau");
    PNODE_REQUIRE(!tab->fsal || d_kbuf, "pnode_cnf_rk_solve_ctl: FSAL tableau without slope buffers");
    PNODE_REQUIRE(ntraj > 0, "pnode_cnf_rk_solve_ctl: bad ntraj");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    PNODE_CUDA_OK(cudaStreamIsCapturing(st, &cap));
    PNODE_REQUIRE(cap == cudaStreamCaptureStatusNone, "pnode_cnf_rk_solve_ctl: the stream is being captured");
    CnfLoopKey k;
    memset(&k, 0, sizeof(k));  // padding bytes take part in the comparison
    k.cnf = *cnf, k.tab = *tab;
    k.ubuf = d_ubuf, k.kbuf = d_kbuf, k.ckpt = d_ckpt_base, k.sol = d_sol, k.ctl = d_ctl, k.work = d_work;
    k.ntraj = ntraj, k.ckpt_step_elems = ckpt_step_elems, k.atol = atol, k.rtol = rtol;
    k.peer_bufs = reinterpret_cast<const unsigned long long *>(d_peer_bufs), k.rank = rank, k.world = world;
    std::lock_guard<std::mutex> lock(g_loop_mutex);
    CnfLoopGraph *hit = nullptr, *victim = &g_loops[0];
    for (auto &g : g_loops) {
        if (g.exec != nullptr && memcmp(&g.key, &k, sizeof(k)) == 0) hit = &g;
        if (g.last_use < victim->last_use) victim = &g;
    }
    if (hit == nullptr) {
        int rc = build_loop_graph(k, *victim);
        if (rc != 0) return rc;
        hit = victim;
    }
    hit->last_use = ++g_loop_clock;
    PNODE_CUDA_OK(cudaGraphLaunch(hit->exec, st));
    return 0;
}

int64_t pnode_cnf_rk_adjoint_work_bytes(const pnode_cnf_desc *cnf) {
    int64_t np = 2 * (int64_t)cnf->hidden * cnf->dim + 4 * cnf->hidden + 4 * cnf->dim;
    return 64 + (int64_t)CNF_MAX_BLOCKS * np * (int64_t)sizeof(double);
}

int pnode_cnf_rk_adjoint_dp(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, int64_t ntraj,
                            const pnode_step *d_sched, int nsteps, int last_slot, const void *d_gout, const void *d_ckpt,
                            void *d_lambda, void *d_mu, void *d_work, const uint64_t *d_peer_bufs, int rank, int world,
                            uint64_t epoch, void *stream) {
    PNODE_REQUIRE(cnf && tab && d_sched && d_work && d_ckpt, "pnode_cnf_rk_adjoint: null argument");
    PNODE_REQUIRE(cnf_shape_ok(cnf->dim, cnf->hidden, tab->s), "pnode_cnf_rk_adjoint: unsupported shape D=%d H=%d s=%d",
                  cnf->dim, cnf->hidden, tab->s);
    PNODE_REQUIRE(world <= 1 || d_peer_bufs == nullptr || (epoch >= 1 && rank >= 0 && rank < world && world <= 64),
                  "pnode_cnf_rk_adjoint_dp: bad rank/world/epoch");
    PeerComm pc{reinterpret_cast<const unsigned long long *>(d_peer_bufs), rank, world, (unsigned long long)epoch};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
#define X(SS)                                                                                                       \
    if (tab->s == SS) {                                                                                             \
        if (cnf->dtype == PNODE_F32)                                                                                \
            return launch_cnf_adjoint<float, SS>(cnf, tab, ntraj, d_sched, nsteps, last_slot, d_gout, d_ckpt,        \
                                                 d_lambda, d_mu, d_work, pc, st);                                   \
        return launch_cnf_adjoint<double, SS>(cnf, tab, ntraj, d_sched, nsteps, last_slot, d_gout, d_ckpt, d_lambda, \
                                              d_mu, d_work, pc, st);                                                \
    }
    PNODE_CNF_STAGES(X)
#undef X
    PNODE_REQUIRE(false, "pnode_cnf_rk_adjoint: no kernel for %d stages", tab->s);
}

int pnode_cnf_rk_adjoint(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, int64_t ntraj,
                         const pnode_step *d_sched, int nsteps, int last_slot, const void *d_gout, const void *d_ckpt,
                         void *d_lambda, void *d_mu, void *d_work, void *stream) {
    return pnode_cnf_rk_adjoint_dp(cnf, tab, ntraj, d_sched, nsteps, last_slot, d_gout, d_ckpt, d_lambda, d_mu, d_work,
                                   nullptr, 0, 1, 0, stream);
}

}  // extern "C"
