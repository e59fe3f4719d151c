// Wide ReLU-MLP right-hand sides (SINODE: examples-sinode/KS/models/imex.py:46-70, Burgers.py:134-160) and their
// vector-Jacobian products as chains of tensor-core sliced products (csrc/umma_gemm.cu), plus the circulant implicit
// operator of the same examples (imex.py:6-44): stencil application and the inverse of shift*I - J built from its
// spectrum (no factorisation).
//
//   forward   X_0 = u;  Z_l = X_l W_l^T + b_l;  X_{l+1} = relu(Z_l) (l < L-1);  f = out_scale * Z_{L-1}
//             per layer: slice X_l by rows (A operand), [slice X_l by columns -> activation set, for dW in the adjoint],
//             one product with bias + ReLU in the epilogue.
//   vjp       G_{L-1} = out_scale * w;  per layer, downwards:
//             mu_W_l += coef * G_l^T X_l   (product of the column-sliced G_l and the kept column-sliced X_l, accumulated
//                                           straight into mu: no per-parameter gradient tensors, no AXPY pass)
//             mu_b_l += coef * colsum(G_l) (by-product of the column slicing)
//             G_{l-1} = (G_l W_l) masked by X_l > 0   (ReLU backward in the epilogue);  J^T w = G_0 W_0
#include <math.h>

#include "common.cuh"
#include "umma.cuh"

namespace pnode {
namespace dmlp {

static inline long long align256(long long x) { return (x + 255) / 256 * 256; }

struct Layout {
    int L, kind, esz, batch;
    int dims[PNODE_DMLP_MAX_LAYERS + 1];
    long long wf[PNODE_DMLP_MAX_LAYERS], wf_exp[PNODE_DMLP_MAX_LAYERS], wb[PNODE_DMLP_MAX_LAYERS],
        wb_exp[PNODE_DMLP_MAX_LAYERS], w_total;
    long long act_xt[PNODE_DMLP_MAX_LAYERS], act_xt_exp[PNODE_DMLP_MAX_LAYERS], act_x[PNODE_DMLP_MAX_LAYERS], act_total;
    long long xs, xs_exp, gs, gs_exp, gt, gt_exp, d0, d1, colpart, work_total;
};

static int make_layout(const pnode_dmlp_desc *d, Layout &lay) {
    PNODE_REQUIRE(d != nullptr, "dense mlp: null descriptor");
    PNODE_REQUIRE(d->nlayers >= 1 && d->nlayers <= PNODE_DMLP_MAX_LAYERS, "dense mlp: %d layers (1..%d supported)",
                  d->nlayers, PNODE_DMLP_MAX_LAYERS);
    PNODE_REQUIRE(d->dtype == PNODE_F32 || d->dtype == PNODE_F64, "dense mlp: dtype %d", d->dtype);
    PNODE_REQUIRE(d->batch >= 1, "dense mlp: empty batch");
    lay.L = d->nlayers;
    lay.kind = d->dtype == PNODE_F64 ? umma::KIND_I8 : umma::KIND_TF32;
    if (d->dtype == PNODE_F64) {  // the dense 8-bit digits bound the reduction length (int32 accumulators)
        int longest = d->batch;
        for (int l = 0; l <= d->nlayers; ++l) longest = d->dims[l] > longest ? d->dims[l] : longest;
        if (longest > PNODE_I8_MAX_K) lay.kind = umma::KIND_I8X;
    }
    lay.esz = d->dtype == PNODE_F64 ? 8 : 4;
    lay.batch = d->batch;
    // every width and the batch are the reduction length of some product; fp64 beyond 16384 uses the 8-digit kind
    const int max_k = d->dtype == PNODE_F64 ? PNODE_I8X_MAX_K : 65536;
    int maxdim = 0;
    for (int l = 0; l <= lay.L; ++l) {
        PNODE_REQUIRE(d->dims[l] >= 1 && d->dims[l] <= max_k, "dense mlp: layer width %d (max %d)", d->dims[l], max_k);
        lay.dims[l] = d->dims[l];
        maxdim = d->dims[l] > maxdim ? d->dims[l] : maxdim;
    }
    PNODE_REQUIRE(d->batch <= max_k, "dense mlp: batch %d exceeds the reduction length of one product (max %d)", d->batch,
                  max_k);
    long long off = 0;
    for (int l = 0; l < lay.L; ++l) {
        const int in = lay.dims[l], out = lay.dims[l + 1];
        lay.wf[l] = off, off += align256(umma::sliced_bytes(lay.kind, out, in));
        lay.wf_exp[l] = off, off += align256(4ll * out);
        lay.wb[l] = off, off += align256(umma::sliced_bytes(lay.kind, in, out));
        lay.wb_exp[l] = off, off += align256(4ll * in);
    }
    lay.w_total = off;
    off = 0;
    for (int l = 0; l < lay.L; ++l) {
        lay.act_xt[l] = off, off += align256(umma::sliced_bytes(lay.kind, lay.dims[l], lay.batch));
        lay.act_xt_exp[l] = off, off += align256(4ll * lay.dims[l]);
        lay.act_x[l] = off;
        if (l > 0) off += align256((long long)lay.batch * lay.dims[l] * lay.esz);
    }
    lay.act_total = off;
    off = 0;
    lay.xs = off, off += align256(umma::sliced_bytes(lay.kind, lay.batch, maxdim));
    lay.xs_exp = off, off += align256(4ll * lay.batch);
    lay.gs = off, off += align256(umma::sliced_bytes(lay.kind, lay.batch, maxdim));
    lay.gs_exp = off, off += align256(4ll * lay.batch);
    lay.gt = off, off += align256(umma::sliced_bytes(lay.kind, maxdim, lay.batch));
    lay.gt_exp = off, off += align256(4ll * maxdim);
    lay.d0 = off, off += align256((long long)lay.batch * maxdim * lay.esz);
    lay.d1 = off, off += align256((long long)lay.batch * maxdim * lay.esz);
    lay.colpart = off, off += align256((long long)((lay.batch + 31) / 32) * maxdim * 8);
    lay.work_total = off;
    return 0;
}

// ---- circulant operator ---------------------------------------------------------------------------------------------
struct Taps {
    int n;
    int off[PNODE_CIRC_MAX_TAPS];
    double coef[PNODE_CIRC_MAX_TAPS];
};

// out[r][i] = sum_d coef[d] x[r][(i -/+ off[d]) mod n]   (J[i][j] = c[(i - j) mod n];  transpose: c[(j - i) mod n])
template <typename T>
__global__ void circ_apply_kernel(const T *x, T *out, int rows, int n, Taps taps, int transpose) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const long long total = (long long)rows * n;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(idx % n);
        const T *xr = x + (idx - i);
        // same association as a direct convolution: accumulate the taps in order
        T acc = 0;
        for (int d = 0; d < taps.n; ++d) {
            int j = transpose ? i + taps.off[d] : i - taps.off[d];
            j %= n;
            if (j < 0) j += n;
            acc += (T)taps.coef[d] * xr[j];
        }
        out[idx] = acc;
    }
}

// Spectrum of A = shift*I - J (circulant, first column a = shift*e0 - c):  lam_k = sum_j a_j w^{jk},  w = exp(-2 pi i / n);
// stores 1 / lam_k.
__global__ void circ_spectrum_kernel(const double *col, int n, double shift, double2 *inv_lam) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    double re = 0.0, im = 0.0, cre = 0.0, cim = 0.0;  // Kahan-compensated sums
    for (int j = 0; j < n; ++j) {
        const double a = (j == 0 ? shift : 0.0) - col[j];
        if (a == 0.0) continue;
        const long long m = ((long long)j * k) % n;
        double s, c;
        sincospi(-2.0 * (double)m / (double)n, &s, &c);
        double y = a * c - cre, t = re + y;
        cre = (t - re) - y, re = t;
        y = a * s - cim, t = im + y;
        cim = (t - im) - y, im = t;
    }
    const double den = re * re + im * im;
    inv_lam[k] = make_double2(re / den, -im / den);
}

// First column of A^-1:  g_m = (1/n) sum_k (1/lam_k) w^{-mk}  (real for a real circulant).
__global__ void circ_inverse_column_kernel(const double2 *inv_lam, int n, double *g) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    double acc = 0.0, comp = 0.0;
    for (int k = 0; k < n; ++k) {
        const long long q = ((long long)m * k) % n;
        double s, c;
        sincospi(2.0 * (double)q / (double)n, &s, &c);
        const double2 v = inv_lam[k];
        const double y = (v.x * c - v.y * s) - comp, t = acc + y;
        comp = (t - acc) - y, acc = t;
    }
    g[m] = acc / (double)n;
}

template <typename T>
__global__ void circ_expand_kernel(const double *g, int n, T *dense) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const long long total = (long long)n * n;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / n), j = (int)(idx % n);
        int d = i - j;
        if (d < 0) d += n;
        dense[idx] = (T)g[d];
    }
}

}  // namespace dmlp
}  // namespace pnode

using namespace pnode;
using dmlp::Layout;

extern "C" {

int64_t pnode_dmlp_weight_bytes(const pnode_dmlp_desc *desc) {
    Layout lay;
    return dmlp::make_layout(desc, lay) ? -1 : lay.w_total;
}
int64_t pnode_dmlp_act_bytes(const pnode_dmlp_desc *desc) {
    Layout lay;
    return dmlp::make_layout(desc, lay) ? -1 : lay.act_total;
}
int64_t pnode_dmlp_work_bytes(const pnode_dmlp_desc *desc) {
    Layout lay;
    return dmlp::make_layout(desc, lay) ? -1 : lay.work_total;
}

int pnode_dmlp_prepare(const pnode_dmlp_desc *desc, void *d_wslices, void *stream) {
    Layout lay;
    if (int rc = dmlp::make_layout(desc, lay)) return rc;
    PNODE_REQUIRE(d_wslices != nullptr, "pnode_dmlp_prepare: null workspace");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *W = (uint8_t *)d_wslices;
    for (int l = 0; l < lay.L; ++l) {
        const int in = lay.dims[l], out = lay.dims[l + 1];
        PNODE_REQUIRE(desc->d_weight[l] != nullptr, "pnode_dmlp_prepare: layer %d has no weight", l);
        if (int rc = umma::slice_both(lay.kind, desc->d_weight[l], in, out, in, W + lay.wf[l], (int *)(W + lay.wf_exp[l]),
                                      W + lay.wb[l], (int *)(W + lay.wb_exp[l]), nullptr, 0.0, nullptr, st))
            return rc;
    }
    return 0;
}

int pnode_dmlp_forward(const pnode_dmlp_desc *desc, const void *d_wslices, const void *d_u, void *d_out, void *d_act,
                       void *d_work, void *stream) {
    Layout lay;
    if (int rc = dmlp::make_layout(desc, lay)) return rc;
    PNODE_REQUIRE(d_wslices && d_u && d_out && d_work, "pnode_dmlp_forward: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t *W = (const uint8_t *)d_wslices;
    uint8_t *act = (uint8_t *)d_act, *work = (uint8_t *)d_work;
    const void *X = d_u;
    for (int l = 0; l < lay.L; ++l) {
        const int in = lay.dims[l], out = lay.dims[l + 1];
        const bool last = l == lay.L - 1;
        if (act) {
            if (int rc = umma::slice_both(lay.kind, X, in, lay.batch, in, work + lay.xs, (int *)(work + lay.xs_exp),
                                          act + lay.act_xt[l], (int *)(act + lay.act_xt_exp[l]), nullptr, 0.0, nullptr, st))
                return rc;
        } else if (int rc = umma::slice_rows(lay.kind, X, in, lay.batch, in, work + lay.xs, (int *)(work + lay.xs_exp), st))
            return rc;
        void *Y = last ? d_out : (act ? (void *)(act + lay.act_x[l + 1]) : (void *)(work + ((l & 1) ? lay.d1 : lay.d0)));
        if (int rc = umma::gemm(lay.kind, work + lay.xs, (const int *)(work + lay.xs_exp), W + lay.wf[l],
                                (const int *)(W + lay.wf_exp[l]), lay.batch, out, in, Y, out, last ? desc->out_scale : 1.0,
                                desc->d_bias[l], last ? 0 : 1, nullptr, 0, 0, st))
            return rc;
        X = Y;
    }
    return 0;
}

int pnode_dmlp_vjp(const pnode_dmlp_desc *desc, const void *d_wslices, const void *d_act, const void *d_w, void *d_vu,
                   void *d_mu, double coef, void *d_work, void *stream) {
    return pnode_dmlp_vjp_ev(desc, d_wslices, d_act, d_w, d_vu, d_mu, coef, d_work, nullptr, stream);
}

int pnode_dmlp_vjp_ev(const pnode_dmlp_desc *desc, const void *d_wslices, const void *d_act, const void *d_w, void *d_vu,
                      void *d_mu, double coef, void *d_work, void *const *layer_events, void *stream) {
    Layout lay;
    if (int rc = dmlp::make_layout(desc, lay)) return rc;
    PNODE_REQUIRE(d_wslices && d_act && d_w && d_work, "pnode_dmlp_vjp: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t *W = (const uint8_t *)d_wslices, *act = (const uint8_t *)d_act;
    uint8_t *work = (uint8_t *)d_work, *mu = (uint8_t *)d_mu;
    const void *G = d_w;
    double gscale = desc->out_scale;
    for (int l = lay.L - 1; l >= 0; --l) {
        const int in = lay.dims[l], out = lay.dims[l + 1];
        const bool need_dx = l > 0 || d_vu != nullptr;
        const bool gw = mu && desc->mu_w_off[l] >= 0, gb = mu && desc->mu_b_off[l] >= 0;
        if (need_dx && (gw || gb)) {
            if (int rc = umma::slice_both(lay.kind, G, out, lay.batch, out, work + lay.gs, (int *)(work + lay.gs_exp),
                                          work + lay.gt, (int *)(work + lay.gt_exp),
                                          gb ? mu + desc->mu_b_off[l] * lay.esz : nullptr, coef * gscale,
                                          (double *)(work + lay.colpart), st))
                return rc;
        } else if (need_dx) {
            if (int rc = umma::slice_rows(lay.kind, G, out, lay.batch, out, work + lay.gs, (int *)(work + lay.gs_exp), st))
                return rc;
        } else if (gw || gb) {
            if (int rc = umma::slice_cols(lay.kind, G, out, lay.batch, out, work + lay.gt, (int *)(work + lay.gt_exp),
                                          gb ? mu + desc->mu_b_off[l] * lay.esz : nullptr, coef * gscale, st))
                return rc;
        }
        if (gw || gb) {
            if (gw)
                if (int rc = umma::gemm(lay.kind, work + lay.gt, (const int *)(work + lay.gt_exp), act + lay.act_xt[l],
                                        (const int *)(act + lay.act_xt_exp[l]), out, in, lay.batch,
                                        mu + desc->mu_w_off[l] * lay.esz, in, coef * gscale, nullptr, 0, nullptr, 0, 1, st))
                    return rc;
        }
        if (layer_events != nullptr && layer_events[l] != nullptr)  // layer l's slice of mu is complete for this call
            PNODE_CUDA_OK(cudaEventRecord(static_cast<cudaEvent_t>(layer_events[l]), st));
        if (l > 0) {
            void *Y = work + ((l & 1) ? lay.d1 : lay.d0);
            if (int rc = umma::gemm(lay.kind, work + lay.gs, (const int *)(work + lay.gs_exp), W + lay.wb[l],
                                    (const int *)(W + lay.wb_exp[l]), lay.batch, in, out, Y, in, gscale, nullptr, 0,
                                    act + lay.act_x[l], in, 0, st))
                return rc;
            G = Y;
            gscale = 1.0;
        } else if (d_vu) {
            if (int rc = umma::gemm(lay.kind, work + lay.gs, (const int *)(work + lay.gs_exp), W + lay.wb[0],
                                    (const int *)(W + lay.wb_exp[0]), lay.batch, in, out, d_vu, in, gscale, nullptr, 0, nullptr,
                                    0, 0, st))
                return rc;
        }
    }
    return 0;
}

int pnode_circulant_apply(const void *d_x, void *d_out, int rows, int n, const int32_t *offsets, const double *coefs,
                          int ntaps, int transpose, int dtype, void *stream) {
    PNODE_REQUIRE(d_x && d_out && d_x != d_out, "pnode_circulant_apply: null or aliased vectors");
    PNODE_REQUIRE(ntaps >= 0 && ntaps <= PNODE_CIRC_MAX_TAPS, "pnode_circulant_apply: %d taps (max %d)", ntaps,
                  PNODE_CIRC_MAX_TAPS);
    PNODE_REQUIRE(rows > 0 && n > 0, "pnode_circulant_apply: empty operand");
    dmlp::Taps taps;
    taps.n = ntaps;
    for (int d = 0; d < ntaps; ++d) taps.off[d] = offsets[d], taps.coef[d] = coefs[d];
    const long long total = (long long)rows * n;
    const int grid = (int)((total + 255) / 256 < 8 * sm_count() ? (total + 255) / 256 : 8 * sm_count());
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == PNODE_F64)
        PNODE_CUDA_OK(pdl::launch_pdl(dmlp::circ_apply_kernel<double>, dim3(grid), dim3(256), 0, st, (const double *)d_x, (double *)d_out, rows, n, taps, transpose));
    else if (dtype == PNODE_F32)
        PNODE_CUDA_OK(pdl::launch_pdl(dmlp::circ_apply_kernel<float>, dim3(grid), dim3(256), 0, st, (const float *)d_x, (float *)d_out, rows, n, taps, transpose));
    else
        PNODE_REQUIRE(false, "pnode_circulant_apply: dtype %d", dtype);
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

int64_t pnode_circulant_work_bytes(int n) { return (int64_t)n * 24 + 256; }

int pnode_circulant_inverse(const double *d_col, int n, double shift, void *d_inverse, int dtype, void *d_work, void *stream) {
    PNODE_REQUIRE(d_col && d_inverse && d_work && n > 0, "pnode_circulant_inverse: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    double2 *inv_lam = (double2 *)d_work;
    double *g = (double *)((uint8_t *)d_work + (size_t)n * 16);
    PNODE_CUDA_OK(pdl::launch_pdl(dmlp::circ_spectrum_kernel, dim3((n + 127) / 128), dim3(128), 0, st, d_col, n, shift, inv_lam));
    PNODE_CUDA_OK(pdl::launch_pdl(dmlp::circ_inverse_column_kernel, dim3((n + 127) / 128), dim3(128), 0, st, inv_lam, n, g));
    const long long total = (long long)n * n;
    const int grid = (int)((total + 255) / 256 < 8 * sm_count() ? (total + 255) / 256 : 8 * sm_count());
    if (dtype == PNODE_F64)
        PNODE_CUDA_OK(pdl::launch_pdl(dmlp::circ_expand_kernel<double>, dim3(grid), dim3(256), 0, st, g, n, (double *)d_inverse));
    else if (dtype == PNODE_F32)
        PNODE_CUDA_OK(pdl::launch_pdl(dmlp::circ_expand_kernel<float>, dim3(grid), dim3(256), 0, st, g, n, (float *)d_inverse));
    else
        PNODE_REQUIRE(false, "pnode_circulant_inverse: dtype %d", dtype);
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
