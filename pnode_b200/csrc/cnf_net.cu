// FFJORD ConcatSquash networks of any depth and width (ffjord-pnode/lib/layers/odefunc.py:53-57,345-385 with an ODEnet of
// L ConcatSquashLinear layers + Softplus, diffeq_layers/basic.py:76-86) and their adjoint in closed form, as chains of
// tensor-core sliced products (csrc/umma_gemm.cu) with small elementwise kernels in between.
//
// Per sample (row vectors), x_0 = z, v_0 = e (Hutchinson probe), tau = t (rounded through float32 when the module does):
//   gamma_l = sigmoid(hgw_l tau + hgb_l),  c_l = hbw_l tau
//   P_l = x_l W_l^T + b_l,  Q_l = v_l W_l^T,  a_l = gamma_l P_l + c_l,  u_l = gamma_l Q_l
//   l < L-1:  x_{l+1} = softplus(a_l),  s_l = sigmoid(a_l),  v_{l+1} = s_l u_l        (s = 1 above the threshold 20)
//   f = a_{L-1},  div = e . u_{L-1} (= e^T J e),  F = (f, -div)
// The tangent v is pushed along with x, so the trace needs no backward pass.  The value and tangent chains are stacked as
// 2B rows: one product [x_l; v_l] W_l^T per layer.
//
// Adjoint stage for w = (w_z, w_l):  abar_{L-1} = w_z,  ubar_{L-1} = -w_l e;  for l = L-1 .. 0:
//   Pbar = gamma abar,  Qbar = gamma ubar
//   W_l += coef [Pbar; Qbar]^T [x_l; v_l]        (product with reduction length 2B, accumulated into mu by the epilogue)
//   b_l += coef sum Pbar,  gammabar = sum (abar P + ubar Q),  cbar = sum abar   (per-CTA partials, fixed-order finalize)
//   [xbar; vbar] = [Pbar; Qbar] W_l
//   l > 0:  abar_{l-1} = s xbar + s(1-s) u_{l-1} vbar,  ubar_{l-1} = s vbar   (s = s_{l-1})
//   l = 0:  J^T w = (xbar_0, 0)
//   hgw += coef gammabar gamma(1-gamma) tau,  hgb += coef gammabar gamma(1-gamma),  hbw += coef cbar tau
// Replaces the reference's evalRHSFunction -> ODEfunc.forward (autograd Hutchinson trace) and, per adjoint stage,
// RHSJacShell.multTranspose / RHSJacPShell.multTranspose (second-order autograd, pnode/petsc_adjoint.py:52-82,341-363).
#include <math.h>

#include "common.cuh"
#include "umma.cuh"

namespace pnode {
namespace cnfnet {

constexpr int ROWS_PER_CTA = 32;  // rows of one column-partial block of the adjoint elementwise kernel
constexpr int COLS_PER_CTA = 128;

static inline long long align256(long long x) { return (x + 255) / 256 * 256; }

struct Layout {
    int L, kind, esz, batch, rows, maxdim, nrb;
    int dims[PNODE_DMLP_MAX_LAYERS + 1];
    long long goff[PNODE_DMLP_MAX_LAYERS], gate_total;  // element offset of layer l's (gamma, c) in a gate block
    long long wf[PNODE_DMLP_MAX_LAYERS], wf_exp[PNODE_DMLP_MAX_LAYERS], wb[PNODE_DMLP_MAX_LAYERS],
        wb_exp[PNODE_DMLP_MAX_LAYERS], w_total;
    long long act_xt[PNODE_DMLP_MAX_LAYERS], act_xt_exp[PNODE_DMLP_MAX_LAYERS], act_pq[PNODE_DMLP_MAX_LAYERS], act_gate,
        act_total;
    long long x, xs, xs_exp, y, gate, g, gs, gs_exp, gt, gt_exp, xbar, part, work_total;
};

static int make_layout(const pnode_cnfnet_desc *d, Layout &lay) {
    PNODE_REQUIRE(d != nullptr, "cnf net: null descriptor");
    PNODE_REQUIRE(d->nlayers >= 1 && d->nlayers <= PNODE_DMLP_MAX_LAYERS, "cnf net: %d layers (1..%d supported)", d->nlayers,
                  PNODE_DMLP_MAX_LAYERS);
    PNODE_REQUIRE(d->dtype == PNODE_F32 || d->dtype == PNODE_F64, "cnf net: dtype %d", d->dtype);
    PNODE_REQUIRE(d->batch >= 1, "cnf net: empty batch");
    PNODE_REQUIRE(d->dims[0] == d->dims[d->nlayers], "cnf net: output width %d differs from the state width %d",
                  d->dims[d->nlayers], d->dims[0]);
    lay.L = d->nlayers;
    lay.batch = d->batch;
    lay.rows = 2 * d->batch;  // value and tangent chains stacked
    lay.esz = d->dtype == PNODE_F64 ? 8 : 4;
    // every width and 2B (the weight gradient's reduction length) are the reduction length of some product
    const int max_k = d->dtype == PNODE_F64 ? PNODE_I8X_MAX_K : 65536;
    PNODE_REQUIRE(lay.rows <= max_k, "cnf net: 2 x batch = %d exceeds the reduction length of one product (max %d)",
                  lay.rows, max_k);
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
    // activation set of one evaluation: column-sliced [x_l; v_l] (weight gradient), [P_l; Q_l] (bias included in P) and the
    // gates -- everything the adjoint stage at the same point reads
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

// X[0:B] = z, X[B:2B] = e
template <typename T>
__global__ void stack_kernel(const T *z, const T *e, T *x, long long n) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        x[i] = z[i];
        x[n + i] = e[i];
    }
}

// hidden layer: y = [x W^T; v W^T] -> y[0:B] += b (P kept for the adjoint), x_next = [softplus(a); s * gamma * Q]
template <typename T>
__global__ void forward_elem_kernel(T *y, const T *bias, const T *gate, T *xnext, int batch, int n) {
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
        xnext[total + i] = s * (g * y[total + i]);
    }
}

// last layer: f = gamma P + c into the z block of out, -e . (gamma Q) into the logp block (one thread per sample: the trace is
// summed in a fixed order)
template <typename T>
__global__ void forward_last_kernel(T *y, const T *bias, const T *gate, const T *e, T *out, int batch, int n) {
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
            div += e[i] * (g * y[off + i]);
        }
        out[off + r] = -div;
    }
}

// G = [gamma abar; gamma ubar] for layer l, and per-CTA column partials part[rb][j] = {sum Pbar, sum (abar P + ubar Q),
// sum abar} over this CTA's ROWS_PER_CTA rows, summed in row order.
//   top (l = L-1): abar = w_z, ubar = -w_l e
//   inner:         (xbar, vbar) of layer l+1's data gradient; abar = s xbar + s(1-s) u vbar, ubar = s vbar (layer l's s, u)
template <typename T>
__global__ void adjoint_elem_kernel(const T *pq, const T *gate, const T *w, const T *e, const T *xbar, int top, T *g,
                                    double *part, int batch, int n) {
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
        const T P = pq[i], Q = pq[off + i];
        T abar, ubar;
        if (top) {
            abar = w[i];
            ubar = -w[off + r] * e[i];
        } else {
            T sp, s;
            softplus_sigmoid(gam * P + c, sp, s);
            const T u = gam * Q, xb = xbar[i], vb = xbar[off + i];
            abar = s * xb + s * (T(1) - s) * u * vb;
            ubar = s * vb;
        }
        const T Pb = gam * abar, Qb = gam * ubar;
        g[i] = Pb;
        g[off + i] = Qb;
        sb += (double)Pb;
        sg += (double)abar * (double)P + (double)ubar * (double)Q;
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

template <typename T>
static int forward(const pnode_cnfnet_desc *d, const Layout &lay, const uint8_t *W, double t, const void *d_u, void *d_out,
                   uint8_t *act, uint8_t *work, cudaStream_t st) {
    const Params<T> p = params_of<T>(d, lay);
    const int B = lay.batch, D = lay.dims[0];
    T *gate = (T *)(act ? act + lay.act_gate : work + lay.gate);
    PNODE_CUDA_OK(pdl::launch_pdl(gate_kernel<T>, dim3(grid_for(lay.maxdim, 256)), dim3(256), 0, st, p, tau_of(d, t), gate));
    T *X = (T *)(work + lay.x);
    PNODE_CUDA_OK(pdl::launch_pdl(stack_kernel<T>, dim3(grid_for((long long)B * D, 256)), dim3(256), 0, st, (const T *)d_u,
                                  (const T *)d->d_e, X, (long long)B * D));
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
                                          p.b[l], gl, X, B, out));
        else
            PNODE_CUDA_OK(pdl::launch_pdl(forward_last_kernel<T>, dim3(grid_for(B, 128)), dim3(128), 0, st, Y, p.b[l], gl,
                                          (const T *)d->d_e, (T *)d_out, B, out));
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
    const T *gate = (const T *)(act + lay.act_gate);
    auto at = [&](long long off) -> T * { return (mu && off >= 0) ? mu + off : nullptr; };
    for (int l = lay.L - 1; l >= 0; --l) {
        const int in = lay.dims[l], out = lay.dims[l + 1];
        const T *pq = (const T *)(act + lay.act_pq[l]), *gl = gate + lay.goff[l];
        PNODE_CUDA_OK(pdl::launch_pdl(adjoint_elem_kernel<T>, dim3((out + COLS_PER_CTA - 1) / COLS_PER_CTA, lay.nrb),
                                      dim3(COLS_PER_CTA), 0, st, pq, gl, (const T *)d_w, (const T *)d->d_e,
                                      (const T *)Xbar, l == lay.L - 1 ? 1 : 0, G, part, B, out));
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
            // the data gradient of the first layer needs the value rows only (v_0 = e is a constant)
            if (l > 0 || d_vu)
                if (int rc = umma::slice_rows(lay.kind, G, out, l > 0 ? lay.rows : B, out, work + lay.gs,
                                              (int *)(work + lay.gs_exp), st))
                    return rc;
        }
        if (gw)
            if (int rc = umma::gemm(lay.kind, work + lay.gt, (const int *)(work + lay.gt_exp), act + lay.act_xt[l],
                                    (const int *)(act + lay.act_xt_exp[l]), out, in, lay.rows, mu + d->mu_w_off[l], in, coef,
                                    nullptr, 0, nullptr, 0, 1, st))
                return rc;
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
    PNODE_REQUIRE(d_wslices && d_u && d_out && d_work && desc->d_e, "pnode_cnfnet_forward: null argument");
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
    PNODE_REQUIRE(d_wslices && d_act && d_w && d_work && desc->d_e, "pnode_cnfnet_vjp: null argument");
    const uint8_t *W = (const uint8_t *)d_wslices, *act = (const uint8_t *)d_act;
    uint8_t *work = (uint8_t *)d_work;
    cudaStream_t st = (cudaStream_t)stream;
    return desc->dtype == PNODE_F64 ? cnfnet::vjp<double>(desc, lay, W, t, act, d_w, d_vu, d_mu, coef, work, st)
                                    : cnfnet::vjp<float>(desc, lay, W, t, act, d_w, d_vu, d_mu, coef, work, st);
}

}  // extern "C"
