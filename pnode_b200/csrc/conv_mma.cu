// Tensor-core evaluator of the convolutional ODE block for GEMM-sized shapes (CIFAR blocks 3 and 4 of
// examples-pnode/models/sqnxt_PETSc.py:70-121: [256,128,8,8], [256,256,4,4]; fp32): every convolution, data gradient and
// weight gradient is an implicit GEMM on the 5th-generation tensor cores (csrc/umma_gemm.cu: TMA + tcgen05.mma + TMEM,
// 3xTF32 so that the 1e-4 parity bar of IEEE fp32 holds).
//
// Inside the block activations are pixel-major ("NHWC") matrices [P = N*H*W][C]:
//   forward layer k   A_k = im2col(relu(bn_{k-1}(z_{k-1})))  -- BatchNorm + ReLU of the previous layer applied while the
//                     operand is gathered and split (hi/lo), never written as a tensor;   z_k = A_k W_k^T + bias_k with the
//                     batch statistics of z_k (per-CTA column sums, fixed order) coming out of the product's epilogue
//   data gradient     g_{k-1} = [y_{k-1} > 0] . (im2col'(dz_k) Wd_k^T),  dz_k = a g_k + b z_k + c (BatchNorm backward folded
//                     into the gather), ReLU mask and the sums of the next BatchNorm backward in the epilogue
//   weight gradient   dW_k = dz_k^T A_k: reduction over the pixels, split over the SMs (split-K), partials combined in a
//                     fixed order straight into mu
// Same contract as csrc/conv_block.cu (include/pnode_b200.h): activation sets kept by the caller let the adjoint skip the
// forward re-evaluation; batch-sharded runs exchange the statistics of the GLOBAL batch over NVLink peer memory inside the
// finalize kernels.
#include "common.cuh"
#include "umma.cuh"

namespace pnode {
namespace cmma {

constexpr int KIND = umma::KIND_TF32;
static inline long long al256(long long x) { return (x + 255) / 256 * 256; }

struct Geom {
    int cin, cout, taps, dir;  // dir 0: 1x1;  1: taps along W (kernel (1,3));  2: taps along H (kernel (3,1))
};

struct Plan {
    int L, N, H, W, world, rank;
    long long P, Pg;
    int mtiles, cmax, kcmax;
    Geom g[PNODE_CONV_MAX_LAYERS];
    long long wf[PNODE_CONV_MAX_LAYERS], wd[PNODE_CONV_MAX_LAYERS], w_total;
    long long z[PNODE_CONV_MAX_LAYERS], bnp[PNODE_CONV_MAX_LAYERS], act_total;
    long long xin, win, A, g0, g1, dzT, AT, part, stats, tot, bwdc, work_total;
    long long goff_w[PNODE_CONV_MAX_LAYERS], goff_b[PNODE_CONV_MAX_LAYERS], goff_gamma[PNODE_CONV_MAX_LAYERS],
        goff_beta[PNODE_CONV_MAX_LAYERS], nparams;
};

// split-K slices of the weight-gradient product of one layer: enough CTAs for two per SM
static int wgrad_slices(const Geom &g, long long P, int *kb_per_split) {
    const int kc = g.taps * g.cin;
    const int tiles = ((g.cout + 127) / 128) * ((kc + 63) / 64);
    int splits = 296 / tiles;
    splits = splits < 1 ? 1 : splits;
    const int kb = umma::split_k_blocks(KIND, (int)P, splits);
    const int total_kb = (int)((P + 31) / 32);
    if (kb_per_split) *kb_per_split = kb;
    return (total_kb + kb - 1) / kb;
}

static int make_plan(const pnode_convblock_desc *d, Plan &p) {
    PNODE_REQUIRE(d != nullptr, "conv mma: null descriptor");
    PNODE_REQUIRE(d->dtype == PNODE_F32, "conv mma: the tensor-core evaluator is fp32 (3xTF32)");
    PNODE_REQUIRE(d->nlayers >= 1 && d->nlayers <= PNODE_CONV_MAX_LAYERS, "conv mma: %d layers", d->nlayers);
    p.L = d->nlayers, p.N = d->N, p.H = d->H, p.W = d->W;
    p.P = (long long)d->N * d->H * d->W;
    PNODE_REQUIRE(p.P >= 1 && p.P <= 65536, "conv mma: %lld pixels (the weight-gradient reduction takes <= 65536)", p.P);
    p.world = d->world > 1 ? d->world : 1;
    p.rank = d->world > 1 ? d->rank : 0;
    p.Pg = (d->world > 1 && d->global_pixels > 0) ? d->global_pixels : p.P;
    p.mtiles = (int)((p.P + 127) / 128);
    p.cmax = 0, p.kcmax = 0;
    long long woff = 0, aoff = 0, goff = 0;
    for (int k = 0; k < p.L; ++k) {
        const pnode_conv_layer &l = d->layer[k];
        Geom &g = p.g[k];
        g.cin = l.cin, g.cout = l.cout;
        if (l.kh == 1 && l.kw == 1 && l.ph == 0 && l.pw == 0)
            g.taps = 1, g.dir = 0;
        else if (l.kh == 1 && l.kw == 3 && l.ph == 0 && l.pw == 1)
            g.taps = 3, g.dir = 1;
        else if (l.kh == 3 && l.kw == 1 && l.ph == 1 && l.pw == 0)
            g.taps = 3, g.dir = 2;
        else
            PNODE_REQUIRE(false, "conv mma: layer %d kernel (%d,%d) padding (%d,%d) unsupported", k, l.kh, l.kw, l.ph, l.pw);
        PNODE_REQUIRE(g.cin % 4 == 0 && g.cout % 4 == 0 && g.cin >= 8 && g.cout >= 8, "conv mma: channel counts %d -> %d", g.cin,
                      g.cout);
        PNODE_REQUIRE(k == 0 || g.cin == p.g[k - 1].cout, "conv mma: layer %d does not chain", k);
        PNODE_REQUIRE(2 * g.cout <= PNODE_PEER_NP_MAX, "conv mma: %d channels exceed the peer exchange slot", g.cout);
        const int kc = g.taps * g.cin, kd = g.taps * g.cout;
        p.cmax = max(p.cmax, max(g.cin, g.cout));
        p.kcmax = max(p.kcmax, max(kc, kd));
        p.wf[k] = woff, woff += al256(umma::sliced_bytes(KIND, g.cout, kc));
        p.wd[k] = woff, woff += al256(umma::sliced_bytes(KIND, g.cin, kd));
        p.z[k] = aoff, aoff += al256(p.P * g.cout * 4);
        p.bnp[k] = aoff, aoff += al256(32ll * g.cout);  // doubles mean, invstd; floats a, b, qa, qb
        p.goff_w[k] = goff, goff += (long long)g.cout * g.cin * g.taps;
        p.goff_b[k] = goff, goff += g.cout;
        p.goff_gamma[k] = goff, goff += g.cout;
        p.goff_beta[k] = goff, goff += g.cout;
    }
    PNODE_REQUIRE(p.g[p.L - 1].cout == p.g[0].cin, "conv mma: the block must map the state onto itself");
    p.w_total = woff, p.act_total = aoff, p.nparams = goff;
    long long off = 0;
    p.xin = off, off += al256(p.P * p.cmax * 4);
    p.win = off, off += al256(p.P * p.cmax * 4);
    p.A = off, off += al256(umma::sliced_bytes(KIND, (int)p.P, p.kcmax));
    p.g0 = off, off += al256(p.P * p.cmax * 4);
    p.g1 = off, off += al256(p.P * p.cmax * 4);
    p.dzT = off, off += al256(umma::sliced_bytes(KIND, p.cmax, (int)p.P));
    p.AT = off, off += al256(umma::sliced_bytes(KIND, p.kcmax, (int)p.P));
    long long part = 0;
    for (int k = 0; k < p.L; ++k)
        part = max(part, (long long)wgrad_slices(p.g[k], p.P, nullptr) * p.g[k].cout * p.g[k].taps * p.g[k].cin * 4);
    p.part = off, off += al256(part);
    p.stats = off, off += al256((long long)p.mtiles * p.cmax * 16);
    p.tot = off, off += al256((4ll + 32) * p.cmax * 8);
    p.bwdc = off, off += al256(3ll * p.cmax * 4);
    p.work_total = off;
    return 0;
}

__device__ __forceinline__ float tf32_hi(float x) {
    uint32_t u = __float_as_uint(x);
    if ((u & 0x7f800000u) == 0x7f800000u) return x;
    u += 0xfffu + ((u >> 13) & 1u);
    return __uint_as_float(u & 0xffffe000u);
}

// ---- layout changes between the caller's NCHW state and the pixel-major matrices ------------------------------------
// dst[n][hw][c] = src[n][c][hw]   (grid: hw tiles, c tiles, n)
__global__ void nchw_to_nhwc_kernel(const float *src, float *dst, int C, int HW) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    __shared__ float t[32][33];
    const int n = blockIdx.z, hw0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const float *s = src + (long long)n * C * HW;
    float *d = dst + (long long)n * C * HW;
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int c = c0 + i, hw = hw0 + threadIdx.x;
        t[i][threadIdx.x] = (c < C && hw < HW) ? s[(long long)c * HW + hw] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int hw = hw0 + i, c = c0 + threadIdx.x;
        if (c < C && hw < HW) d[(long long)hw * C + c] = t[threadIdx.x][i];
    }
}

// Output pass of the block: k[n][c][hw] = relu(a[c] z[n][hw][c] + b[c]);  out = base_coef * base + k_coef * k.
__global__ void act_out_kernel(const float *z, const float *a, const float *b, int C, int HW, float *kout, float *out,
                               const float *base, float base_coef, float k_coef) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    __shared__ float t[32][33];
    const int n = blockIdx.z, hw0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const long long img = (long long)n * C * HW;
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int hw = hw0 + i, c = c0 + threadIdx.x;
        float v = 0.f;
        if (c < C && hw < HW) v = fmaxf(fmaf(a[c], z[img + (long long)hw * C + c], b[c]), 0.f);
        t[i][threadIdx.x] = v;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int c = c0 + i, hw = hw0 + threadIdx.x;
        if (c < C && hw < HW) {
            const long long o = img + (long long)c * HW + hw;
            const float kv = t[threadIdx.x][i];
            if (kout) kout[o] = kv;
            if (out) out[o] = base ? fmaf(k_coef, kv, base_coef * base[o]) : k_coef * kv;
        }
    }
}

// g[p][c] = w[n][c][hw] * [a[c] z[p][c] + b[c] > 0]  (cotangent of the block's output through its last ReLU), and the
// per-128-pixel partial sums of the BatchNorm backward: stats[tile][c] = {sum g, sum g * zhat}, zhat = qa[c] z + qb[c].
// grid: (P/128 tiles, c tiles); a tile never straddles... images may: HW is a divisor or a multiple of 32.
__global__ void top_grad_kernel(const float *w, const float *z, const float *a, const float *b, const float *qa,
                                const float *qb, int C, int HW, long long P, float *g, double *stats) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    __shared__ float t[32][33];
    __shared__ double s1[8][33], s2[8][33];
    const int c0 = blockIdx.y * 32;
    double acc1 = 0.0, acc2 = 0.0;  // lane = channel c0 + threadIdx.x, this thread's pixels
    for (int sub = 0; sub < 4; ++sub) {
        const long long p0 = (long long)blockIdx.x * 128 + sub * 32;
        for (int i = threadIdx.y; i < 32; i += 8) {  // read NCHW with lanes along the pixels
            const int c = c0 + i;
            const long long p = p0 + threadIdx.x;
            float v = 0.f;
            if (c < C && p < P) v = w[(p / HW) * (long long)C * HW + (long long)c * HW + (p % HW)];
            t[i][threadIdx.x] = v;
        }
        __syncthreads();
        for (int i = threadIdx.y; i < 32; i += 8) {  // write pixel-major with lanes along the channels
            const long long p = p0 + i;
            const int c = c0 + threadIdx.x;
            if (c < C && p < P) {
                const float zv = z[p * C + c];
                const float gv = fmaf(a[c], zv, b[c]) > 0.f ? t[threadIdx.x][i] : 0.f;
                g[p * C + c] = gv;
                acc1 += (double)gv;
                acc2 += (double)gv * ((double)qa[c] * (double)zv + (double)qb[c]);
            }
        }
        __syncthreads();
    }
    s1[threadIdx.y][threadIdx.x] = acc1;
    s2[threadIdx.y][threadIdx.x] = acc2;
    __syncthreads();
    if (threadIdx.y == 0 && c0 + threadIdx.x < C) {
        for (int r = 1; r < 8; ++r) acc1 += s1[r][threadIdx.x], acc2 += s2[r][threadIdx.x];
        double *dst = stats + ((long long)blockIdx.x * C + c0 + threadIdx.x) * 2;
        dst[0] = acc1, dst[1] = acc2;
    }
}

// ---- operand gathers --------------------------------------------------------------------------------------------------
enum { SRC_RAW = 0, SRC_ACT = 1, SRC_DZ = 2 };

struct Gather {
    const float *src;   // RAW: values;  ACT: z of the previous layer;  DZ: g of this layer
    const float *src2;  // DZ: z of this layer
    const float *a, *b, *c;  // per-channel coefficients: ACT relu(a z + b);  DZ a g + b z + c
    int mode, C, taps, dir, sign, H, W;
    long long P;
};

__device__ __forceinline__ float gather_value(const Gather &G, long long q, int c) {
    if (G.mode == SRC_RAW) return G.src[q * G.C + c];
    if (G.mode == SRC_ACT) return fmaxf(fmaf(G.a[c], G.src[q * G.C + c], G.b[c]), 0.f);
    return fmaf(G.a[c], G.src[q * G.C + c], fmaf(G.b[c], G.src2[q * G.C + c], G.c[c]));
}

// source pixel of tap t for destination pixel p, or -1 outside the image (zero padding)
__device__ __forceinline__ long long tap_source(const Gather &G, long long p, int t) {
    if (G.taps == 1) return p;
    const int s = (t - 1) * G.sign;
    const int hw = (int)(p % ((long long)G.H * G.W));
    if (G.dir == 1) {
        const int w = hw % G.W + s;
        return (w >= 0 && w < G.W) ? p + s : -1;
    }
    const int h = hw / G.W + s;
    return (h >= 0 && h < G.H) ? p + (long long)s * G.W : -1;
}

// A[s][p][t*C + c] (row-major operand of the products over channels), 4 channels per thread.
__global__ void gather_rows_kernel(Gather G, float *out, long long pitch_f, long long slice_f) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const int c4n = G.C / 4;
    const long long total = G.P * G.taps * c4n;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % c4n) * 4;
        const int t = (int)((idx / c4n) % G.taps);
        const long long p = idx / ((long long)c4n * G.taps);
        const long long q = tap_source(G, p, t);
        float4 hi = make_float4(0.f, 0.f, 0.f, 0.f), lo = hi;
        if (q >= 0) {
            float v[4];
            if (G.mode == SRC_RAW) {
                const float4 x = *reinterpret_cast<const float4 *>(G.src + q * G.C + c);
                v[0] = x.x, v[1] = x.y, v[2] = x.z, v[3] = x.w;
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) v[i] = gather_value(G, q, c + i);
            }
            hi = make_float4(tf32_hi(v[0]), tf32_hi(v[1]), tf32_hi(v[2]), tf32_hi(v[3]));
            lo = make_float4(v[0] - hi.x, v[1] - hi.y, v[2] - hi.z, v[3] - hi.w);
        }
        float *o = out + p * pitch_f + (long long)t * G.C + c;
        *reinterpret_cast<float4 *>(o) = hi;
        *reinterpret_cast<float4 *>(o + slice_f) = lo;
    }
}

// AT[s][t*C + c][p] (operand of the products over pixels): 32 pixels x 32 channels per block and tap.
__global__ void gather_cols_kernel(Gather G, float *out, long long pitch_f, long long slice_f) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    __shared__ float th[32][33], tl[32][33];
    const int t = blockIdx.z, c0 = blockIdx.y * 32;
    const long long p0 = (long long)blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += 8) {
        const long long p = p0 + i;
        const int c = c0 + threadIdx.x;
        float v = 0.f;
        if (p < G.P && c < G.C) {
            const long long q = tap_source(G, p, t);
            if (q >= 0) v = gather_value(G, q, c);
        }
        const float hi = tf32_hi(v);
        th[i][threadIdx.x] = hi;
        tl[i][threadIdx.x] = v - hi;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int c = c0 + i;
        const long long p = p0 + threadIdx.x;
        if (c < G.C && p < G.P) {
            float *o = out + ((long long)t * G.C + c) * pitch_f + p;
            o[0] = th[threadIdx.x][i];
            o[slice_f] = tl[threadIdx.x][i];
        }
    }
}

// ---- weights ------------------------------------------------------------------------------------------------------------
// wf[s][co][t*cin + ci] = W[co][ci][t]  (forward / weight-gradient layout);  wd[s][ci][t*cout + co] = W[co][ci][t] (data gradient)
__global__ void weight_operands_kernel(const float *w, int cin, int cout, int taps, float *wf, long long wf_pitch,
                                       long long wf_slice, float *wd, long long wd_pitch, long long wd_slice) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const int total = cout * cin * taps;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int t = idx % taps, ci = (idx / taps) % cin, co = idx / (taps * cin);
        const float v = w[idx], hi = tf32_hi(v), lo = v - hi;
        float *f = wf + (long long)co * wf_pitch + t * cin + ci;
        f[0] = hi, f[wf_slice] = lo;
        float *d = wd + (long long)ci * wd_pitch + t * cout + co;
        d[0] = hi, d[wd_slice] = lo;
    }
}

// Totals of the per-row-block partial sums, fixed order: RG threads per channel take contiguous ranges of the row blocks,
// their sums are combined in range order.  tot[c] = sum of [.][c][0], tot[C + c] = sum of [.][c][1].  All threads of the block.
template <int RGMAX>
__device__ void reduce_partials(const double *partials, int mtiles, int C, double *tot, double *scratch /* [2][RGMAX][C] */) {
    // One block sums [mtiles][C][2] partials.  The block is alone on its SM and every load is an L2 round trip, so the loads
    // of a range are issued eight row blocks at a time before they are added (in range order), and the per-range sums go
    // through shared memory when they fit (32 KB) instead of the global scratch: 22 us -> a few us per layer at C = 128.
    constexpr int SH = 2048;
    __shared__ double sh[2 * SH];
    const bool in_smem = C <= SH;
    const int RG = in_smem ? max(1, min(RGMAX, SH / C)) : RGMAX;
    double *s1buf = in_smem ? sh : scratch, *s2buf = in_smem ? sh + RG * C : scratch + (long long)RG * C;
    const int per = (mtiles + RG - 1) / RG;
    for (int i = threadIdx.x; i < C * RG; i += blockDim.x) {
        const int c = i % C, g = i / C;
        const int m0 = g * per, m1 = min(mtiles, m0 + per);
        double s1 = 0.0, s2 = 0.0;
        for (int m = m0; m < m1; m += 8) {
            double a[8], b[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const bool in = m + u < m1;
                const double *q = partials + ((long long)(in ? m + u : m) * C + c) * 2;
                a[u] = in ? q[0] : 0.0;
                b[u] = in ? q[1] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) s1 += a[u], s2 += b[u];
        }
        s1buf[(long long)g * C + c] = s1;
        s2buf[(long long)g * C + c] = s2;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        double s1 = 0.0, s2 = 0.0;
        for (int g = 0; g < RG; ++g) s1 += s1buf[(long long)g * C + c], s2 += s2buf[(long long)g * C + c];
        tot[c] = s1, tot[C + c] = s2;
    }
    __syncthreads();
}

// ---- BatchNorm bookkeeping (one block; the cross-GPU exchange of common.cuh needs all threads of ONE block) ----------
struct BnFwd {
    const double *partials;  // [mtiles][C][2]
    int mtiles, C;
    double count;            // pixels of the global batch
    const float *gamma, *beta;
    float *running_mean, *running_var;
    long long *num_batches_tracked;
    double eps, momentum;
    double *mean, *invstd;   // activation set
    float *a, *b, *qa, *qb;
    double *tot, *tot_global;  // scratch [2C] each
    double *scratch;           // [2][16][C]
    int update_running;
};

__global__ void bn_forward_finalize_kernel(BnFwd B, PeerComm pc) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const int C = B.C;
    reduce_partials<16>(B.partials, B.mtiles, C, B.tot, B.scratch);
    const double *tot = B.tot;
    if (pc.world > 1 && pc.peer_bufs) {
        peer_allreduce_and_store<double>(B.tot, 2 * C, pc, B.tot_global);
        __syncthreads();
        tot = B.tot_global;
    }
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const double mean = tot[c] / B.count;
        double var = tot[C + c] / B.count - mean * mean;
        var = var > 0.0 ? var : 0.0;
        const double invstd = rsqrt(var + B.eps);
        const double a = (double)B.gamma[c] * invstd;
        B.mean[c] = mean, B.invstd[c] = invstd;
        B.a[c] = (float)a, B.b[c] = (float)((double)B.beta[c] - mean * a);
        B.qa[c] = (float)invstd, B.qb[c] = (float)(-mean * invstd);
        if (B.update_running && B.running_mean) {
            const double unbiased = B.count > 1.0 ? var * B.count / (B.count - 1.0) : var;
            B.running_mean[c] = (float)((1.0 - B.momentum) * (double)B.running_mean[c] + B.momentum * mean);
            B.running_var[c] = (float)((1.0 - B.momentum) * (double)B.running_var[c] + B.momentum * unbiased);
        }
    }
    if (threadIdx.x == 0 && B.update_running && B.num_batches_tracked) *B.num_batches_tracked += 1;
}

struct BnBwd {
    const double *partials;  // [mtiles][C][2] = {sum g, sum g zhat}
    int mtiles, C;
    double count;
    const float *gamma;
    const double *mean, *invstd;
    float *ca, *cb, *cc;     // dz = ca g + cb z + cc
    float *ggamma, *gbeta, *gbias;  // gradient slots (NULL: not wanted)
    double coef;
    int accumulate, contribute;    // contribute == 0: another rank reports the (global) affine gradients
    double *tot, *tot_global, *scratch;
    // adjoint of an evaluation whose activation set was kept: the module's re-evaluation would have advanced the BatchNorm
    // buffers once more (SURVEY.md H4.iv) -- done here from the stored statistics instead of in a launch of its own
    int advance_running;
    double eps, momentum;
    float *running_mean, *running_var;
    long long *num_batches_tracked;
};

__global__ void bn_backward_finalize_kernel(BnBwd B, PeerComm pc) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const int C = B.C;
    if (B.advance_running) {
        if (B.running_mean) {
            for (int c = threadIdx.x; c < C; c += blockDim.x) {
                const double var = fmax(1.0 / (B.invstd[c] * B.invstd[c]) - B.eps, 0.0);
                const double unbiased = B.count > 1.0 ? var * B.count / (B.count - 1.0) : var;
                B.running_mean[c] = (float)((1.0 - B.momentum) * (double)B.running_mean[c] + B.momentum * B.mean[c]);
                B.running_var[c] = (float)((1.0 - B.momentum) * (double)B.running_var[c] + B.momentum * unbiased);
            }
        }
        if (threadIdx.x == 0 && B.num_batches_tracked) *B.num_batches_tracked += 1;
    }
    reduce_partials<16>(B.partials, B.mtiles, C, B.tot, B.scratch);
    const double *tot = B.tot;
    if (pc.world > 1 && pc.peer_bufs) {
        peer_allreduce_and_store<double>(B.tot, 2 * C, pc, B.tot_global);
        __syncthreads();
        tot = B.tot_global;
    }
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const double S1 = tot[c], S2 = tot[C + c];
        const double m1 = S1 / B.count, m2 = S2 / B.count;
        const double a = (double)B.gamma[c] * B.invstd[c];
        B.ca[c] = (float)a;
        B.cb[c] = (float)(-a * m2 * B.invstd[c]);
        B.cc[c] = (float)(-a * m1 + a * m2 * B.invstd[c] * B.mean[c]);
        if (B.ggamma) {
            const double dg = B.contribute ? S2 : 0.0, db = B.contribute ? S1 : 0.0;
            if (B.accumulate) {
                B.ggamma[c] += (float)(B.coef * dg);
                B.gbeta[c] += (float)(B.coef * db);
            } else {
                B.ggamma[c] = (float)dg;
                B.gbeta[c] = (float)db;
                B.gbias[c] = 0.f;  // a convolution bias feeding a BatchNorm has an exactly zero gradient
            }
        }
    }
}

// grads_w[co][ci][t] (+)= coef * sum_s part[s][co][t*cin + ci]: 8 lanes per entry take contiguous ranges of the split-K
// slices, combined in lane order (fixed order => bit-reproducible)
__global__ void wgrad_reduce_kernel(const float *part, int splits, int cout, int cin, int taps, float *gw, double coef,
                                    int accumulate) {
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const int kc = cin * taps, total = cout * kc;
    const int sub = threadIdx.x & 7;
    const int idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    double s = 0.0;
    if (idx < total) {
        const int per = (splits + 7) / 8, k0 = sub * per, k1 = min(splits, k0 + per);
        for (int k = k0; k < k1; ++k) s += (double)part[(long long)k * total + idx];
    }
    double sum = 0.0;
#pragma unroll
    for (int l = 0; l < 8; ++l) sum += __shfl_sync(0xffffffffu, s, (threadIdx.x & 24) + l);
    if (idx < total && sub == 0) {
        const int co = idx / kc, r = idx % kc, t = r / cin, ci = r % cin;
        float *dst = gw + ((long long)co * cin + ci) * taps + t;
        *dst = accumulate ? (float)((double)*dst + coef * sum) : (float)sum;
    }
}

// ---- host orchestration -----------------------------------------------------------------------------------------------
static PeerComm peer_of(const pnode_convblock_desc *d, unsigned long long epoch) {
    PeerComm pc;
    pc.peer_bufs = (d->world > 1) ? reinterpret_cast<const unsigned long long *>(d->d_peer_bufs) : nullptr;
    pc.rank = d->rank, pc.world = d->world > 1 ? d->world : 1, pc.epoch = epoch;
    return pc;
}

static int launch_gather_rows(const Gather &G, uint8_t *A, int kc, cudaStream_t st) {
    const long long pitch_f = umma::pitch_bytes(KIND, kc) / 4, slice_f = G.P * pitch_f;
    const long long total = G.P * G.taps * (G.C / 4);
    const int grid = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    PNODE_CUDA_OK(pdl::launch_pdl(gather_rows_kernel, dim3(grid), dim3(256), 0, st, G, reinterpret_cast<float *>(A), pitch_f, slice_f));
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

static int launch_gather_cols(const Gather &G, uint8_t *AT, cudaStream_t st) {
    const long long pitch_f = umma::pitch_bytes(KIND, (int)G.P) / 4, slice_f = (long long)G.taps * G.C * pitch_f;
    dim3 grid((unsigned)((G.P + 31) / 32), (G.C + 31) / 32, G.taps);
    PNODE_CUDA_OK(pdl::launch_pdl(gather_cols_kernel, dim3(grid), dim3(32, 8), 0, st, G, reinterpret_cast<float *>(AT), pitch_f, slice_f));
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

static Gather base_gather(const Plan &p, const Geom &g, int channels, int sign) {
    Gather G{};
    G.C = channels, G.taps = g.taps, G.dir = g.dir, G.sign = sign, G.H = p.H, G.W = p.W, G.P = p.P;
    return G;
}

struct Bnp {
    double *mean, *invstd;
    float *a, *b, *qa, *qb;
};
static Bnp bnp_of(const Plan &p, uint8_t *act, int k) {
    const int C = p.g[k].cout;
    uint8_t *b = act + p.bnp[k];
    Bnp r;
    r.mean = reinterpret_cast<double *>(b), r.invstd = r.mean + C;
    r.a = reinterpret_cast<float *>(b + 16ll * C), r.b = r.a + C, r.qa = r.b + C, r.qb = r.qa + C;
    return r;
}

static int forward_impl(const pnode_convblock_desc *d, const Plan &p, const uint8_t *W, const float *x, uint8_t *act,
                        uint8_t *work, unsigned long long epoch, cudaStream_t st) {
    const int HW = p.H * p.W, C0 = p.g[0].cin;
    float *xin = reinterpret_cast<float *>(work + p.xin);
    PNODE_CUDA_OK(pdl::launch_pdl(nchw_to_nhwc_kernel, dim3(dim3((HW + 31) / 32, (C0 + 31) / 32, p.N)), dim3(32, 8), 0, st, x, xin, C0, HW));
    for (int k = 0; k < p.L; ++k) {
        const Geom &g = p.g[k];
        const pnode_conv_layer &l = d->layer[k];
        const int kc = g.taps * g.cin;
        Gather G = base_gather(p, g, g.cin, +1);
        if (k == 0) {
            G.mode = SRC_RAW, G.src = xin;
        } else {
            const Bnp prev = bnp_of(p, act, k - 1);
            G.mode = SRC_ACT, G.src = reinterpret_cast<const float *>(act + p.z[k - 1]), G.a = prev.a, G.b = prev.b;
        }
        if (int rc = launch_gather_rows(G, work + p.A, kc, st)) return rc;
        umma::Epilogue ep{};
        ep.C = act + p.z[k], ep.ldc = g.cout, ep.alpha = 1.0, ep.bias = l.d_bias;
        ep.stats = reinterpret_cast<double *>(work + p.stats), ep.stat_mode = 1;
        if (int rc = umma::gemm_ex(KIND, work + p.A, W + p.wf[k], (int)p.P, g.cout, kc, ep, st)) return rc;
        const Bnp cur = bnp_of(p, act, k);
        BnFwd B{};
        B.partials = ep.stats, B.mtiles = p.mtiles, B.C = g.cout, B.count = (double)p.Pg;
        B.gamma = (const float *)l.d_gamma, B.beta = (const float *)l.d_beta;
        B.running_mean = (float *)l.d_running_mean, B.running_var = (float *)l.d_running_var;
        B.num_batches_tracked = (long long *)l.d_num_batches_tracked;
        B.eps = l.eps, B.momentum = l.momentum, B.mean = cur.mean, B.invstd = cur.invstd;
        B.a = cur.a, B.b = cur.b, B.qa = cur.qa, B.qb = cur.qb;
        B.tot = reinterpret_cast<double *>(work + p.tot), B.tot_global = B.tot + 2 * p.cmax, B.update_running = 1;
        B.scratch = B.tot + 4 * p.cmax;
        PNODE_CUDA_OK(pdl::launch_pdl(bn_forward_finalize_kernel, dim3(1), dim3(1024), 0, st, B, peer_of(d, epoch + k)));
    }
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace cmma
}  // namespace pnode

using namespace pnode;
using cmma::Plan;

extern "C" {

int64_t pnode_convmma_act_bytes(const pnode_convblock_desc *desc) {
    Plan p;
    return cmma::make_plan(desc, p) ? -1 : p.act_total;
}
int64_t pnode_convmma_work_bytes(const pnode_convblock_desc *desc) {
    Plan p;
    return cmma::make_plan(desc, p) ? -1 : p.work_total;
}
int64_t pnode_convmma_weight_bytes(const pnode_convblock_desc *desc) {
    Plan p;
    return cmma::make_plan(desc, p) ? -1 : p.w_total;
}
int64_t pnode_convmma_param_count(const pnode_convblock_desc *desc) {
    Plan p;
    return cmma::make_plan(desc, p) ? -1 : p.nparams;
}

int pnode_convmma_prepare(const pnode_convblock_desc *desc, void *d_wbuf, void *stream) {
    Plan p;
    if (int rc = cmma::make_plan(desc, p)) return rc;
    PNODE_REQUIRE(d_wbuf != nullptr, "pnode_convmma_prepare: null workspace");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *W = (uint8_t *)d_wbuf;
    for (int k = 0; k < p.L; ++k) {
        const cmma::Geom &g = p.g[k];
        const int kc = g.taps * g.cin, kd = g.taps * g.cout;
        const long long fp = umma::pitch_bytes(cmma::KIND, kc) / 4, dp = umma::pitch_bytes(cmma::KIND, kd) / 4;
        PNODE_CUDA_OK(pdl::launch_pdl(cmma::weight_operands_kernel, dim3((g.cout * kc + 255) / 256), dim3(256), 0, st, (const float *)desc->layer[k].d_weight, g.cin, g.cout, g.taps, (float *)(W + p.wf[k]), fp, (long long)g.cout * fp,
            (float *)(W + p.wd[k]), dp, (long long)g.cin * dp));
    }
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

int pnode_convmma_forward(const pnode_convblock_desc *desc, const void *d_wbuf, const void *d_x, void *d_out,
                          const void *d_base, double base_coef, double k_coef, void *d_k, void *d_act, void *d_work,
                          void *stream) {
    Plan p;
    if (int rc = cmma::make_plan(desc, p)) return rc;
    PNODE_REQUIRE(d_wbuf && d_x && d_act && d_work && (d_out || d_k), "pnode_convmma_forward: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *act = (uint8_t *)d_act, *work = (uint8_t *)d_work;
    if (int rc = cmma::forward_impl(desc, p, (const uint8_t *)d_wbuf, (const float *)d_x, act, work, desc->epoch, st)) return rc;
    const int HW = p.H * p.W, CL = p.g[p.L - 1].cout;
    const cmma::Bnp last = cmma::bnp_of(p, act, p.L - 1);
    PNODE_CUDA_OK(pdl::launch_pdl(cmma::act_out_kernel, dim3(dim3((HW + 31) / 32, (CL + 31) / 32, p.N)), dim3(32, 8), 0, st, (const float *)(act + p.z[p.L - 1]), last.a, last.b, CL, HW, (float *)d_k, (float *)d_out, (const float *)d_base,
        (float)base_coef, (float)k_coef));
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

int pnode_convmma_vjp(const pnode_convblock_desc *desc, const void *d_wbuf, const void *d_x, const void *d_w, void *d_vu,
                      void *d_grads, double coef, int accumulate, void *d_act, int act_valid, void *d_work, void *stream) {
    Plan p;
    if (int rc = cmma::make_plan(desc, p)) return rc;
    PNODE_REQUIRE(d_wbuf && d_x && d_w && d_act && d_work, "pnode_convmma_vjp: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t *W = (const uint8_t *)d_wbuf;
    uint8_t *act = (uint8_t *)d_act, *work = (uint8_t *)d_work;
    float *grads = (float *)d_grads;
    const int HW = p.H * p.W, C0 = p.g[0].cin;
    unsigned long long epoch = desc->epoch;
    float *xin = reinterpret_cast<float *>(work + p.xin);
    if (!act_valid) {
        if (int rc = cmma::forward_impl(desc, p, W, (const float *)d_x, act, work, epoch, st)) return rc;
        epoch += p.L;
    } else {
        // no re-evaluation: the module's forward would still have advanced the BatchNorm buffers once (done by the
        // backward-finalize launch of each layer below)
        PNODE_CUDA_OK(pdl::launch_pdl(cmma::nchw_to_nhwc_kernel, dim3(dim3((HW + 31) / 32, (C0 + 31) / 32, p.N)), dim3(32, 8), 0, st, (const float *)d_x, xin, C0, HW));
    }
    double *stats = reinterpret_cast<double *>(work + p.stats);
    double *tot = reinterpret_cast<double *>(work + p.tot);
    float *ca = reinterpret_cast<float *>(work + p.bwdc), *cb = ca + p.cmax, *cc = cb + p.cmax;
    float *gbuf[2] = {reinterpret_cast<float *>(work + p.g0), reinterpret_cast<float *>(work + p.g1)};
    int cur = 0;
    // cotangent through the last ReLU, pixel-major, with the sums of the last BatchNorm's backward
    {
        const int k = p.L - 1, C = p.g[k].cout;
        const cmma::Bnp b = cmma::bnp_of(p, act, k);
        PNODE_CUDA_OK(pdl::launch_pdl(cmma::top_grad_kernel, dim3(dim3(p.mtiles, (C + 31) / 32)), dim3(32, 8), 0, st, (const float *)d_w, (const float *)(act + p.z[k]), b.a, b.b, b.qa, b.qb, C, HW, p.P, gbuf[cur], stats));
    }
    for (int k = p.L - 1; k >= 0; --k) {
        const cmma::Geom &g = p.g[k];
        const pnode_conv_layer &l = desc->layer[k];
        const cmma::Bnp b = cmma::bnp_of(p, act, k);
        const float *zk = (const float *)(act + p.z[k]);
        cmma::BnBwd B{};
        B.partials = stats, B.mtiles = p.mtiles, B.C = g.cout, B.count = (double)p.Pg, B.gamma = (const float *)l.d_gamma;
        B.mean = b.mean, B.invstd = b.invstd, B.ca = ca, B.cb = cb, B.cc = cc;
        if (grads) B.ggamma = grads + p.goff_gamma[k], B.gbeta = grads + p.goff_beta[k], B.gbias = grads + p.goff_b[k];
        B.coef = coef, B.accumulate = accumulate, B.contribute = (p.world == 1 || p.rank == 0) ? 1 : 0;
        B.tot = tot, B.tot_global = tot + 2 * p.cmax, B.scratch = tot + 4 * p.cmax;
        B.advance_running = act_valid ? 1 : 0, B.eps = l.eps, B.momentum = l.momentum;
        B.running_mean = (float *)l.d_running_mean, B.running_var = (float *)l.d_running_var;
        B.num_batches_tracked = (long long *)l.d_num_batches_tracked;
        PNODE_CUDA_OK(pdl::launch_pdl(cmma::bn_backward_finalize_kernel, dim3(1), dim3(1024), 0, st, B, cmma::peer_of(desc, epoch + (p.L - 1 - k))));
        const int kc = g.taps * g.cin, kd = g.taps * g.cout;
        // dz_k = ca g_k + cb z_k + cc, formed inside the gathers
        cmma::Gather D = cmma::base_gather(p, g, g.cout, -1);
        D.mode = cmma::SRC_DZ, D.src = gbuf[cur], D.src2 = zk, D.a = ca, D.b = cb, D.c = cc;
        if (grads) {
            cmma::Gather DT = D;
            DT.taps = 1, DT.dir = 0;
            if (int rc = cmma::launch_gather_cols(DT, work + p.dzT, st)) return rc;
            cmma::Gather AT = cmma::base_gather(p, g, g.cin, +1);
            if (k == 0) {
                AT.mode = cmma::SRC_RAW, AT.src = xin;
            } else {
                const cmma::Bnp prev = cmma::bnp_of(p, act, k - 1);
                AT.mode = cmma::SRC_ACT, AT.src = (const float *)(act + p.z[k - 1]), AT.a = prev.a, AT.b = prev.b;
            }
            if (int rc = cmma::launch_gather_cols(AT, work + p.AT, st)) return rc;
            umma::Epilogue ep{};
            ep.C = work + p.part, ep.ldc = kc, ep.alpha = 1.0;
            const int nsplit = cmma::wgrad_slices(g, p.P, &ep.kb_per_split);
            ep.split_stride = (long long)g.cout * kc;
            if (int rc = umma::gemm_ex(cmma::KIND, work + p.dzT, work + p.AT, g.cout, kc, (int)p.P, ep, st)) return rc;
            PNODE_CUDA_OK(pdl::launch_pdl(cmma::wgrad_reduce_kernel, dim3((g.cout * kc * 8 + 255) / 256), dim3(256), 0, st, (const float *)(work + p.part), nsplit, g.cout,
                                                                               g.cin, g.taps, grads + p.goff_w[k], coef,
                                                                               accumulate));
        }
        if (k > 0 || d_vu) {
            if (int rc = cmma::launch_gather_rows(D, work + p.A, kd, st)) return rc;
            umma::Epilogue ep{};
            ep.alpha = 1.0, ep.ldc = g.cin;
            if (k > 0) {
                const cmma::Bnp prev = cmma::bnp_of(p, act, k - 1);
                ep.C = gbuf[cur ^ 1];
                ep.mask = act + p.z[k - 1], ep.ldmask = g.cin, ep.mask_a = prev.a, ep.mask_b = prev.b;
                ep.stats = stats, ep.stat_mode = 2, ep.q_a = prev.qa, ep.q_b = prev.qb;
            } else {
                ep.C = work + p.win;
            }
            if (int rc = umma::gemm_ex(cmma::KIND, work + p.A, W + p.wd[k], (int)p.P, g.cin, kd, ep, st)) return rc;
            cur ^= 1;
        }
    }
    if (d_vu)  // pixel-major -> the caller's NCHW: the transpose kernel with the roles of C and HW exchanged
        PNODE_CUDA_OK(pdl::launch_pdl(cmma::nchw_to_nhwc_kernel, dim3(dim3((C0 + 31) / 32, (HW + 31) / 32, p.N)), dim3(32, 8), 0, st, (const float *)(work + p.win), (float *)d_vu, HW, C0));
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // extern "C"
