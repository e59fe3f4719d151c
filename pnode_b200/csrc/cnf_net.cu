// FFJORD ConcatSquash networks of any depth and width (ffjord-pnode/lib/layers/odefunc.py:53-57,345-385 with an ODEnet of
// L ConcatSquashLinear layers + Softplus, diffeq_layers/basic.py:76-86) and their adjoint in closed form, as chains of
// tensor-core sliced products (csrc/umma_gemm.cu) with small elementwise kernels in between.
//
// Per sample (row vectors), x_0 = z, tau = t (rounded through float32 when the module does), and nchain tangent chains
// k = 0 .. nchain-1: one chain v_0 = e (Hutchinson probe, divergence_approx) or D chains v_0^(k) = e_k (the unit vectors,
// exact trace, divergence_bf):
//   gamma_l = sigmoid(hgw_l tau + hgb_l),  c_l = hbw_l tau
//   P_l = x_l W_l^T + b_l,  Q_l^(k) = v_l^(k) W_l^T,  a_l = gamma_l P_l + c_l,  u_l^(k) = gamma_l Q_l^(k)
//   l < L-1:  x_{l+1} = softplus(a_l),  s_l = sigmoid(a_l),  v_{l+1}^(k) = s_l u_l^(k)    (s = 1 above the threshold 20)
//   f = a_{L-1},  div = e . u_{L-1} (= e^T J e)  or  sum_k u_{L-1}^(k)[k] (= tr J, summed in k order),  F = (f, -div)
// The tangents are pushed along with x, so the trace needs no backward pass.  The value and tangent chains are stacked
// chain-major as R = (1 + nchain) B rows [x; v^(0); ...; v^(nchain-1)]: one product per layer.
//
// Adjoint stage for w = (w_z, w_l):  abar_{L-1} = w_z,  ubar_{L-1}^(k) = -w_l e (Hutchinson) or -w_l e_k (exact);
// for l = L-1 .. 0:
//   Pbar = gamma abar,  Qbar^(k) = gamma ubar^(k)
//   W_l += coef [Pbar; Qbar^(0); ...]^T [x_l; v_l^(0); ...]   (product with reduction length R, accumulated into mu by the
//                                                              epilogue; in fp32 with D chains, split-K slices of about B
//                                                              rows combined in slice order, see make_layout)
//   b_l += coef sum Pbar,  gammabar = sum (abar P + sum_k ubar^(k) Q^(k)),  cbar = sum abar   (per-CTA partials,
//                                                                                          fixed-order finalize)
//   [xbar; vbar^(0); ...] = [Pbar; Qbar^(0); ...] W_l
//   l > 0:  abar_{l-1} = s xbar + s(1-s) sum_k u_{l-1}^(k) vbar^(k),  ubar_{l-1}^(k) = s vbar^(k)   (s = s_{l-1})
//   l = 0:  J^T w = (xbar_0, 0)
//   hgw += coef gammabar gamma(1-gamma) tau,  hgb += coef gammabar gamma(1-gamma),  hbw += coef cbar tau
// Replaces the reference's evalRHSFunction -> ODEfunc.forward (autograd Hutchinson trace) and, per adjoint stage,
// RHSJacShell.multTranspose / RHSJacPShell.multTranspose (second-order autograd, pnode/petsc_adjoint.py:52-82,341-363).
#include <math.h>

#include <algorithm>

#include "common.cuh"
#include "umma.cuh"

namespace pnode {
namespace cnfnet {

constexpr int ROWS_PER_CTA = 32;  // rows of one column-partial block of the adjoint elementwise kernel
constexpr int COLS_PER_CTA = 128;

static inline long long align256(long long x) { return (x + 255) / 256 * 256; }

struct Layout {
    int L, kind, esz, batch, nchain, rows, maxdim, nrb, wsplit, wsplit_kb;
    int dims[PNODE_DMLP_MAX_LAYERS + 1];
    long long goff[PNODE_DMLP_MAX_LAYERS], gate_total;  // element offset of layer l's (gamma, c) in a gate block
    long long wf[PNODE_DMLP_MAX_LAYERS], wf_exp[PNODE_DMLP_MAX_LAYERS], wb[PNODE_DMLP_MAX_LAYERS],
        wb_exp[PNODE_DMLP_MAX_LAYERS], w_total;
    long long act_xt[PNODE_DMLP_MAX_LAYERS], act_xt_exp[PNODE_DMLP_MAX_LAYERS], act_pq[PNODE_DMLP_MAX_LAYERS], act_gate,
        act_total;
    long long x, xs, xs_exp, y, gate, g, gs, gs_exp, gt, gt_exp, xbar, part, wpart, work_total;
};

static int make_layout(const pnode_cnfnet_desc *d, Layout &lay) {
    PNODE_REQUIRE(d != nullptr, "cnf net: null descriptor");
    PNODE_REQUIRE(d->nlayers >= 1 && d->nlayers <= PNODE_DMLP_MAX_LAYERS, "cnf net: %d layers (1..%d supported)", d->nlayers,
                  PNODE_DMLP_MAX_LAYERS);
    PNODE_REQUIRE(d->dtype == PNODE_F32 || d->dtype == PNODE_F64, "cnf net: dtype %d", d->dtype);
    PNODE_REQUIRE(d->batch >= 1, "cnf net: empty batch");
    PNODE_REQUIRE(d->trace == 0 || d->trace == 1, "cnf net: trace kind %d (0: Hutchinson, 1: exact)", d->trace);
    PNODE_REQUIRE(d->dims[0] == d->dims[d->nlayers], "cnf net: output width %d differs from the state width %d",
                  d->dims[d->nlayers], d->dims[0]);
    lay.L = d->nlayers;
    lay.batch = d->batch;
    lay.nchain = d->trace ? d->dims[0] : 1;
    lay.esz = d->dtype == PNODE_F64 ? 8 : 4;
    // every width and (1 + nchain) B (the weight gradient's reduction length) are the reduction length of some product
    const int max_k = d->dtype == PNODE_F64 ? PNODE_I8X_MAX_K : 65536;
    const long long rows = (1ll + lay.nchain) * d->batch;  // value and tangent chains stacked
    PNODE_REQUIRE(rows <= max_k, "cnf net: (1 + %d chains) x batch = %lld exceeds the reduction length of one product (max %d)",
                  lay.nchain, rows, max_k);
    lay.rows = (int)rows;
    int longest = lay.rows, maxdim = 0;
    for (int l = 0; l <= lay.L; ++l) {
        PNODE_REQUIRE(d->dims[l] >= 1 && d->dims[l] <= max_k, "cnf net: layer width %d (max %d)", d->dims[l], max_k);
        lay.dims[l] = d->dims[l];
        maxdim = d->dims[l] > maxdim ? d->dims[l] : maxdim;
        longest = d->dims[l] > longest ? d->dims[l] : longest;
    }
    lay.maxdim = maxdim;
    lay.kind = d->dtype == PNODE_F64 ? (longest > PNODE_I8_MAX_K ? umma::KIND_I8X : umma::KIND_I8) : umma::KIND_TF32;
    lay.nrb = (lay.batch + ROWS_PER_CTA - 1) / ROWS_PER_CTA;
    // fp32 with D chains: one fp32 accumulation over all (D + 1) B rows of the weight gradient loses digits in proportion to
    // its length (miniboone, 44000 rows: 3e-4 relative against fp64), so the product is cut into split-K slices of about B
    // rows -- the reduction length of one chain -- and the slices are added in order, in double, into mu.  int8 digits
    // accumulate exactly, and the Hutchinson trace keeps its single product of 2B rows.
    lay.wsplit = 1, lay.wsplit_kb = 0;
    if (lay.kind == umma::KIND_TF32 && lay.nchain > 1) {
        const int total_kb = (lay.rows + 31) / 32;  // K blocks of 32 floats
        lay.wsplit_kb = umma::split_k_blocks(lay.kind, lay.rows, 1 + lay.nchain);
        lay.wsplit = (total_kb + lay.wsplit_kb - 1) / lay.wsplit_kb;
    }
    long long maxwt = 0;  // largest weight matrix
    for (int l = 0; l < lay.L; ++l) maxwt = std::max(maxwt, (long long)lay.dims[l] * lay.dims[l + 1]);
    long long goff = 0;
    for (int l = 0; l < lay.L; ++l) lay.goff[l] = goff, goff += 2ll * lay.dims[l + 1];
    lay.gate_total = goff;
    long long off = 0;
    for (int l = 0; l < lay.L; ++l) {
        const int in = lay.dims[l], out = lay.dims[l + 1];
        lay.wf[l] = off, off += align256(umma::sliced_bytes(lay.kind, out, in));
        lay.wf_exp[l] = off, off += align256(4ll * out);
        lay.wb[l] = off, off += align256(umma::sliced_bytes(lay.kind, in, out));
        lay.wb_exp[l] = off, off += align256(4ll * in);
    }
    lay.w_total = off;
    // activation set of one evaluation: column-sliced [x_l; v_l^(k)] (weight gradient), [P_l; Q_l^(k)] (bias included in P)
    // and the gates -- everything the adjoint stage at the same point reads
    off = 0;
    for (int l = 0; l < lay.L; ++l) {
        lay.act_xt[l] = off, off += align256(umma::sliced_bytes(lay.kind, lay.dims[l], lay.rows));
        lay.act_xt_exp[l] = off, off += align256(4ll * lay.dims[l]);
        lay.act_pq[l] = off, off += align256((long long)lay.rows * lay.dims[l + 1] * lay.esz);
    }
    lay.act_gate = off, off += align256(lay.gate_total * lay.esz);
    lay.act_total = off;
    off = 0;
    const long long stacked = align256((long long)lay.rows * maxdim * lay.esz);
    lay.x = off, off += stacked;
    lay.xs = off, off += align256(umma::sliced_bytes(lay.kind, lay.rows, maxdim));
    lay.xs_exp = off, off += align256(4ll * lay.rows);
    lay.y = off, off += stacked;
    lay.gate = off, off += align256(lay.gate_total * lay.esz);
    lay.g = off, off += stacked;
    lay.gs = off, off += align256(umma::sliced_bytes(lay.kind, lay.rows, maxdim));
    lay.gs_exp = off, off += align256(4ll * lay.rows);
    lay.gt = off, off += align256(umma::sliced_bytes(lay.kind, maxdim, lay.rows));
    lay.gt_exp = off, off += align256(4ll * maxdim);
    lay.xbar = off, off += stacked;
    lay.part = off, off += align256((long long)lay.nrb * maxdim * 3 * 8);
    lay.wpart = off, off += lay.wsplit_kb > 0 ? align256((long long)lay.wsplit * maxwt * 4) : 0;
    lay.work_total = off;
    return 0;
}

static inline double tau_of(const pnode_cnfnet_desc *d, double t) { return d->t_f32 ? (double)(float)t : t; }

static inline int grid_for(long long n, int block) {
    const long long g = (n + block - 1) / block, cap = 8ll * sm_count();
    return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

template <typename T>
__device__ __forceinline__ T sigmoid_(T a) {
    return T(1) / (T(1) + exp(-a));
}

// torch.nn.Softplus(beta=1, threshold=20): identity above the threshold, where its derivative is exactly 1 and its second
// derivative exactly 0
template <typename T>
__device__ __forceinline__ void softplus_sigmoid(T a, T &sp, T &s) {
    if (a > T(20)) {
        sp = a, s = T(1);
    } else {
        sp = log1p(exp(a)), s = sigmoid_(a);
    }
}

template <typename T>
struct Params {
    const T *w[PNODE_DMLP_MAX_LAYERS], *b[PNODE_DMLP_MAX_LAYERS], *hbw[PNODE_DMLP_MAX_LAYERS], *hgw[PNODE_DMLP_MAX_LAYERS],
        *hgb[PNODE_DMLP_MAX_LAYERS];
    long long goff[PNODE_DMLP_MAX_LAYERS];
    int dims[PNODE_DMLP_MAX_LAYERS + 1];
    int L;
};

template <typename T>
static Params<T> params_of(const pnode_cnfnet_desc *d, const Layout &lay) {
    Params<T> p = {};
    p.L = lay.L;
    for (int l = 0; l <= lay.L; ++l) p.dims[l] = lay.dims[l];
    for (int l = 0; l < lay.L; ++l) {
        p.w[l] = (const T *)d->d_weight[l], p.b[l] = (const T *)d->d_bias[l], p.hbw[l] = (const T *)d->d_hyper_bias[l];
        p.hgw[l] = (const T *)d->d_gate_weight[l], p.hgb[l] = (const T *)d->d_gate_bias[l];
        p.goff[l] = lay.goff[l];
    }
    return p;
}

// gate[goff[l] + j] = gamma_l[j], gate[goff[l] + dims[l+1] + j] = c_l[j], for every layer: t arrives as an argument, so
// a recorded CUDA graph re-reads nothing from the host
template <typename T>
__global__ void gate_kernel(Params<T> p, double tau, T *gate) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const T tt = (T)tau;
    for (int l = 0; l < p.L; ++l) {
        const int n = p.dims[l + 1];
        for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
            gate[p.goff[l] + j] = sigmoid_(p.hgw[l][j] * tt + p.hgb[l][j]);
            gate[p.goff[l] + n + j] = p.hbw[l][j] * tt;
        }
    }
}

// X[0:B] = z, then chain k's B rows X[(1+k)B : (2+k)B] = e (Hutchinson, one chain) or the unit vector e_k (exact, e = null)
template <typename T>
__global__ void stack_kernel(const T *z, const T *e, T *x, long long n, int dim, int nchain) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const long long total = (1ll + nchain) * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long blk = i / n, q = i - blk * n;
        x[i] = blk == 0 ? z[q] : e ? e[q] : T(q % dim == blk - 1 ? 1 : 0);
    }
}

// hidden layer: y = [x W^T; v^(k) W^T ...] -> y[0:B] += b (P kept for the adjoint),
// x_next = [softplus(a); s * gamma * Q^(0); ...; s * gamma * Q^(nchain-1)]
template <typename T>
__global__ void forward_elem_kernel(T *y, const T *bias, const T *gate, T *xnext, int batch, int n, int nchain) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const long long total = (long long)batch * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(i % n);
        const T P = y[i] + bias[j];
        y[i] = P;
        const T g = gate[j];
        T sp, s;
        softplus_sigmoid(g * P + gate[n + j], sp, s);
        xnext[i] = sp;
        for (int k = 1; k <= nchain; ++k) xnext[k * total + i] = s * (g * y[k * total + i]);
    }
}

// last layer: f = gamma P + c into the z block of out, -div into the logp block with div = e . (gamma Q) (Hutchinson) or
// sum_k gamma[k] Q^(k)[k] (exact, e = null).  One thread per sample: the trace is summed in a fixed order.
template <typename T>
__global__ void forward_last_kernel(T *y, const T *bias, const T *gate, const T *e, T *out, int batch, int n, int nchain) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const long long off = (long long)batch * n;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < batch; r += gridDim.x * blockDim.x) {
        T div = 0;
        for (int j = 0; j < n; ++j) {
            const long long i = (long long)r * n + j;
            const T P = y[i] + bias[j];
            y[i] = P;
            const T g = gate[j];
            out[i] = g * P + gate[n + j];
            if (e) div += e[i] * (g * y[off + i]);
        }
        if (!e)
            for (int k = 0; k < nchain; ++k) div += gate[k] * y[(1 + k) * off + (long long)r * n + k];
        out[off + r] = -div;
    }
}

// G = [gamma abar; gamma ubar^(0); ...] for layer l, and per-CTA column partials part[rb][j] = {sum Pbar,
// sum (abar P + sum_k ubar^(k) Q^(k)), sum abar} over this CTA's ROWS_PER_CTA rows, summed in row order (chains in k order).
//   top (l = L-1): abar = w_z, ubar^(k) = -w_l e (Hutchinson) or -w_l e_k (exact, e = null)
//   inner:         (xbar, vbar^(k)) of layer l+1's data gradient; abar = s xbar + s(1-s) sum_k u^(k) vbar^(k),
//                  ubar^(k) = s vbar^(k) (layer l's s, u)
template <typename T>
__global__ void adjoint_elem_kernel(const T *pq, const T *gate, const T *w, const T *e, const T *xbar, int top, T *g,
                                    double *part, int batch, int n, int nchain) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const long long off = (long long)batch * n;
    const T gam = gate[j], c = gate[n + j];
    double sb = 0.0, sg = 0.0, sc = 0.0;
    const int r0 = blockIdx.y * ROWS_PER_CTA, r1 = r0 + ROWS_PER_CTA < batch ? r0 + ROWS_PER_CTA : batch;
    for (int r = r0; r < r1; ++r) {
        const long long i = (long long)r * n + j;
        const T P = pq[i];
        T s = T(1), acc = T(0);  // acc = s(1-s) sum_k u^(k) vbar^(k)
        if (!top) {
            T sp;
            softplus_sigmoid(gam * P + c, sp, s);
        }
        const T ss = s * (T(1) - s);
        double sq = 0.0;  // sum_k ubar^(k) Q^(k)
        for (int k = 1; k <= nchain; ++k) {
            const long long ik = k * off + i;
            const T Q = pq[ik];
            T ubar;
            if (top) {
                ubar = e ? -w[off + r] * e[i] : (j == k - 1 ? -w[off + r] : T(0));
            } else {
                const T vb = xbar[ik];
                acc += ss * (gam * Q) * vb;
                ubar = s * vb;
            }
            g[ik] = gam * ubar;
            sq += (double)ubar * (double)Q;
        }
        const T abar = top ? w[i] : s * xbar[i] + acc;
        const T Pb = gam * abar;
        g[i] = Pb;
        sb += (double)Pb;
        sg += (double)abar * (double)P + sq;
        sc += (double)abar;
    }
    double *pp = part + ((long long)blockIdx.y * n + j) * 3;
    pp[0] = sb, pp[1] = sg, pp[2] = sc;
}

// mu += coef * (bias, hyper-bias, gate weight, gate bias gradients) of one layer, partials summed in row-block order
template <typename T>
__global__ void finalize_kernel(const double *part, int nrb, int n, const T *gate, double tau, double coef, T *mu_b,
                                T *mu_hbw, T *mu_hgw, T *mu_hgb) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    double sb = 0.0, sg = 0.0, sc = 0.0;
    for (int rb = 0; rb < nrb; ++rb) {
        const double *pp = part + ((long long)rb * n + j) * 3;
        sb += pp[0], sg += pp[1], sc += pp[2];
    }
    const double gam = (double)gate[j], gg = sg * gam * (1.0 - gam);
    if (mu_b) mu_b[j] += (T)(coef * sb);
    if (mu_hbw) mu_hbw[j] += (T)(coef * sc * tau);
    if (mu_hgw) mu_hgw[j] += (T)(coef * gg * tau);
    if (mu_hgb) mu_hgb[j] += (T)(coef * gg);
}

// mu_w += coef * sum_z part[z] over the split-K slices of the fp32 weight gradient, added in slice order in double
__global__ void wgrad_reduce_kernel(const float *part, int nsplit, long long n, double coef, float *mu_w) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int z = 0; z < nsplit; ++z) s += (double)part[z * n + i];
        mu_w[i] = (float)((double)mu_w[i] + coef * s);
    }
}

template <typename T>
static int forward(const pnode_cnfnet_desc *d, const Layout &lay, const uint8_t *W, double t, const void *d_u, void *d_out,
                   uint8_t *act, uint8_t *work, cudaStream_t st) {
    const Params<T> p = params_of<T>(d, lay);
    const int B = lay.batch, D = lay.dims[0];
    T *gate = (T *)(act ? act + lay.act_gate : work + lay.gate);
    PNODE_CUDA_OK(pdl::launch_pdl(gate_kernel<T>, dim3(grid_for(lay.maxdim, 256)), dim3(256), 0, st, p, tau_of(d, t), gate));
    T *X = (T *)(work + lay.x);
    const T *e = d->trace ? nullptr : (const T *)d->d_e;
    PNODE_CUDA_OK(pdl::launch_pdl(stack_kernel<T>, dim3(grid_for((long long)lay.rows * D, 256)), dim3(256), 0, st,
                                  (const T *)d_u, e, X, (long long)B * D, D, lay.nchain));
    for (int l = 0; l < lay.L; ++l) {
        const int in = lay.dims[l], out = lay.dims[l + 1];
        if (act) {
            if (int rc = umma::slice_both(lay.kind, X, in, lay.rows, in, work + lay.xs, (int *)(work + lay.xs_exp),
                                          act + lay.act_xt[l], (int *)(act + lay.act_xt_exp[l]), nullptr, 0.0, nullptr, st))
                return rc;
        } else if (int rc = umma::slice_rows(lay.kind, X, in, lay.rows, in, work + lay.xs, (int *)(work + lay.xs_exp), st))
            return rc;
        T *Y = (T *)(act ? act + lay.act_pq[l] : work + lay.y);
        if (int rc = umma::gemm(lay.kind, work + lay.xs, (const int *)(work + lay.xs_exp), W + lay.wf[l],
                                (const int *)(W + lay.wf_exp[l]), lay.rows, out, in, Y, out, 1.0, nullptr, 0, nullptr, 0, 0, st))
            return rc;
        const T *gl = gate + lay.goff[l];
        if (l < lay.L - 1)
            PNODE_CUDA_OK(pdl::launch_pdl(forward_elem_kernel<T>, dim3(grid_for((long long)B * out, 256)), dim3(256), 0, st, Y,
                                          p.b[l], gl, X, B, out, lay.nchain));
        else
            PNODE_CUDA_OK(pdl::launch_pdl(forward_last_kernel<T>, dim3(grid_for(B, 128)), dim3(128), 0, st, Y, p.b[l], gl, e,
                                          (T *)d_out, B, out, lay.nchain));
    }
    return 0;
}

template <typename T>
static int vjp(const pnode_cnfnet_desc *d, const Layout &lay, const uint8_t *W, double t, const uint8_t *act, const void *d_w,
               void *d_vu, void *d_mu, double coef, uint8_t *work, cudaStream_t st) {
    const int B = lay.batch;
    const double tau = tau_of(d, t);
    T *mu = (T *)d_mu, *G = (T *)(work + lay.g), *Xbar = (T *)(work + lay.xbar);
    double *part = (double *)(work + lay.part);
    const T *gate = (const T *)(act + lay.act_gate), *e = d->trace ? nullptr : (const T *)d->d_e;
    auto at = [&](long long off) -> T * { return (mu && off >= 0) ? mu + off : nullptr; };
    for (int l = lay.L - 1; l >= 0; --l) {
        const int in = lay.dims[l], out = lay.dims[l + 1];
        const T *pq = (const T *)(act + lay.act_pq[l]), *gl = gate + lay.goff[l];
        PNODE_CUDA_OK(pdl::launch_pdl(adjoint_elem_kernel<T>, dim3((out + COLS_PER_CTA - 1) / COLS_PER_CTA, lay.nrb),
                                      dim3(COLS_PER_CTA), 0, st, pq, gl, (const T *)d_w, e, (const T *)Xbar,
                                      l == lay.L - 1 ? 1 : 0, G, part, B, out, lay.nchain));
        T *mb = at(d->mu_b_off[l]), *mhb = at(d->mu_hbw_off[l]), *mgw = at(d->mu_hgw_off[l]), *mgb = at(d->mu_hgb_off[l]);
        if (mb || mhb || mgw || mgb)
            PNODE_CUDA_OK(pdl::launch_pdl(finalize_kernel<T>, dim3((out + 127) / 128), dim3(128), 0, st, (const double *)part,
                                          lay.nrb, out, gl, tau, coef, mb, mhb, mgw, mgb));
        const bool gw = at(d->mu_w_off[l]) != nullptr;
        if (l > 0 && gw) {
            if (int rc = umma::slice_both(lay.kind, G, out, lay.rows, out, work + lay.gs, (int *)(work + lay.gs_exp),
                                          work + lay.gt, (int *)(work + lay.gt_exp), nullptr, 0.0, nullptr, st))
                return rc;
        } else {
            if (gw)
                if (int rc = umma::slice_cols(lay.kind, G, out, lay.rows, out, work + lay.gt, (int *)(work + lay.gt_exp),
                                              nullptr, 0.0, st))
                    return rc;
            // the data gradient of the first layer needs the value rows only (v_0 = e or e_k is a constant)
            if (l > 0 || d_vu)
                if (int rc = umma::slice_rows(lay.kind, G, out, l > 0 ? lay.rows : B, out, work + lay.gs,
                                              (int *)(work + lay.gs_exp), st))
                    return rc;
        }
        if (gw && lay.wsplit_kb > 0) {
            umma::Epilogue ep{};
            ep.C = work + lay.wpart, ep.ldc = in, ep.alpha = 1.0;
            ep.ea = (const int *)(work + lay.gt_exp), ep.eb = (const int *)(act + lay.act_xt_exp[l]);
            ep.kb_per_split = lay.wsplit_kb, ep.split_stride = (long long)out * in;
            if (int rc = umma::gemm_ex(lay.kind, work + lay.gt, act + lay.act_xt[l], out, in, lay.rows, ep, st)) return rc;
            PNODE_CUDA_OK(pdl::launch_pdl(wgrad_reduce_kernel, dim3(grid_for((long long)out * in, 256)), dim3(256), 0, st,
                                          (const float *)(work + lay.wpart), lay.wsplit, (long long)out * in, coef,
                                          (float *)(mu + d->mu_w_off[l])));
        } else if (gw) {
            if (int rc = umma::gemm(lay.kind, work + lay.gt, (const int *)(work + lay.gt_exp), act + lay.act_xt[l],
                                    (const int *)(act + lay.act_xt_exp[l]), out, in, lay.rows, mu + d->mu_w_off[l], in, coef,
                                    nullptr, 0, nullptr, 0, 1, st))
                return rc;
        }
        if (l > 0) {
            if (int rc = umma::gemm(lay.kind, work + lay.gs, (const int *)(work + lay.gs_exp), W + lay.wb[l],
                                    (const int *)(W + lay.wb_exp[l]), lay.rows, in, out, Xbar, in, 1.0, nullptr, 0, nullptr, 0,
                                    0, st))
                return rc;
        } else if (d_vu) {
            if (int rc = umma::gemm(lay.kind, work + lay.gs, (const int *)(work + lay.gs_exp), W + lay.wb[0],
                                    (const int *)(W + lay.wb_exp[0]), B, in, out, d_vu, in, 1.0, nullptr, 0, nullptr, 0, 0, st))
                return rc;
            PNODE_CUDA_OK(cudaMemsetAsync((T *)d_vu + (long long)B * in, 0, (size_t)B * sizeof(T), st));  // logp feeds nothing
        }
    }
    return 0;
}

}  // namespace cnfnet
}  // namespace pnode

using namespace pnode;
using cnfnet::Layout;

extern "C" {

int64_t pnode_cnfnet_weight_bytes(const pnode_cnfnet_desc *desc) {
    Layout lay;
    return cnfnet::make_layout(desc, lay) ? -1 : lay.w_total;
}
int64_t pnode_cnfnet_act_bytes(const pnode_cnfnet_desc *desc) {
    Layout lay;
    return cnfnet::make_layout(desc, lay) ? -1 : lay.act_total;
}
int64_t pnode_cnfnet_work_bytes(const pnode_cnfnet_desc *desc) {
    Layout lay;
    return cnfnet::make_layout(desc, lay) ? -1 : lay.work_total;
}

int pnode_cnfnet_prepare(const pnode_cnfnet_desc *desc, void *d_wslices, void *stream) {
    Layout lay;
    if (int rc = cnfnet::make_layout(desc, lay)) return rc;
    PNODE_REQUIRE(d_wslices != nullptr, "pnode_cnfnet_prepare: null workspace");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *W = (uint8_t *)d_wslices;
    for (int l = 0; l < lay.L; ++l) {
        const int in = lay.dims[l], out = lay.dims[l + 1];
        PNODE_REQUIRE(desc->d_weight[l] && desc->d_bias[l] && desc->d_hyper_bias[l] && desc->d_gate_weight[l] &&
                          desc->d_gate_bias[l],
                      "pnode_cnfnet_prepare: layer %d lacks a parameter", l);
        if (int rc = umma::slice_both(lay.kind, desc->d_weight[l], in, out, in, W + lay.wf[l], (int *)(W + lay.wf_exp[l]),
                                      W + lay.wb[l], (int *)(W + lay.wb_exp[l]), nullptr, 0.0, nullptr, st))
            return rc;
    }
    return 0;
}

int pnode_cnfnet_forward(const pnode_cnfnet_desc *desc, const void *d_wslices, double t, const void *d_u, void *d_out,
                         void *d_act, void *d_work, void *stream) {
    Layout lay;
    if (int rc = cnfnet::make_layout(desc, lay)) return rc;
    PNODE_REQUIRE(d_wslices && d_u && d_out && d_work && (desc->d_e || desc->trace), "pnode_cnfnet_forward: null argument");
    PNODE_REQUIRE(d_u != d_out, "pnode_cnfnet_forward: aliased state and output");
    const uint8_t *W = (const uint8_t *)d_wslices;
    uint8_t *act = (uint8_t *)d_act, *work = (uint8_t *)d_work;
    cudaStream_t st = (cudaStream_t)stream;
    return desc->dtype == PNODE_F64 ? cnfnet::forward<double>(desc, lay, W, t, d_u, d_out, act, work, st)
                                    : cnfnet::forward<float>(desc, lay, W, t, d_u, d_out, act, work, st);
}

int pnode_cnfnet_vjp(const pnode_cnfnet_desc *desc, const void *d_wslices, double t, const void *d_act, const void *d_w,
                     void *d_vu, void *d_mu, double coef, void *d_work, void *stream) {
    Layout lay;
    if (int rc = cnfnet::make_layout(desc, lay)) return rc;
    PNODE_REQUIRE(d_wslices && d_act && d_w && d_work && (desc->d_e || desc->trace), "pnode_cnfnet_vjp: null argument");
    const uint8_t *W = (const uint8_t *)d_wslices, *act = (const uint8_t *)d_act;
    uint8_t *work = (uint8_t *)d_work;
    cudaStream_t st = (cudaStream_t)stream;
    return desc->dtype == PNODE_F64 ? cnfnet::vjp<double>(desc, lay, W, t, act, d_w, d_vu, d_mu, coef, work, st)
                                    : cnfnet::vjp<float>(desc, lay, W, t, act, d_w, d_vu, d_mu, coef, work, st);
}

}  // extern "C"
