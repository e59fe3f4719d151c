// Convolutional ODE-block right-hand side and its vector-Jacobian products as hand-written sm_100a kernels
// (BASELINE config 4: the SqueezeNext block of /root/reference/examples-pnode/models/sqnxt_PETSc.py:70-121 -- a chain of
// relu(bn_k(conv_k(.))) with 1x1, (1,3) and (3,1) stride-1 "same" convolutions and nn.BatchNorm2d in TRAIN mode).
//
// What it replaces: the arithmetic of the reference's evalRHSFunction (pnode/petsc_adjoint.py:393-412: one forward of the
// module) and RHSJacShell.multTranspose (52-82: one forward re-evaluation + one autograd backward) for this module family.
//
// Design (SURVEY.md section 8d: the first two blocks are HBM-bound, AI 6-12 flop/B; channel counts are 8..32, far too small
// for MMA tiles, so these are CUDA-core FMA kernels whose job is to touch every activation once):
//   * every layer is ONE kernel: it reads the raw output z_{k-1} of the previous convolution, applies that layer's
//     BatchNorm scale/shift + ReLU in registers on load, convolves, adds the bias, writes z_k, and accumulates the
//     per-channel sum / sum of squares of z_k for the NEXT BatchNorm in its epilogue.  relu(bn(z)) is never materialised
//     between layers: per layer the HBM traffic is (C_in + C_out) scalars per pixel, the lower bound of section 8d.
//   * batch statistics are accumulated EXACTLY: every CTA adds its partial sums into 128-bit fixed-point accumulators
//     (two 64-bit integer atomics with carry; integer addition is associative, so the totals are bit-reproducible whatever
//     the order the CTAs finish in).  There is no "last CTA" reduction tail and no separate finalise launch: the kernels
//     that CONSUME a layer's statistics derive mean / inv-std / scale / shift from the accumulators in their prologue (one
//     L2 round trip, overlapped with staging the weights), and CTA (0,0) of the first consumer updates running_mean /
//     running_var / num_batches_tracked like nn.BatchNorm2d.  These grids are a single wave of latency-bound CTAs, so the
//     number of dependent memory round trips per kernel is what is minimised.
//   * thread = 4 consecutive pixels of one image row (one 16-byte access per channel) x RC output channels; weights of the
//     CTA's channel tile sit in shared memory and are read as broadcast LDS.128; horizontal taps come from the neighbouring
//     lanes by warp shuffle, vertical taps from the rows above / below (L1 hits); the loads of the next group of input
//     channels are issued before the FMAs of the current one (register double buffer).
//   * the backward of a layer is two kernels over the same inputs (g_k = dL/dy_k, z_k, z_{k-1}): a data-gradient kernel --
//     the same convolution kernel with the BatchNorm+ReLU backward  dz = c0 [y>0] g + c1 (z - mean) + c2  applied on load,
//     flipped taps / transposed weights, and the NEXT layer's backward reductions (sum [y>0] g, sum [y>0] g xhat) in its
//     epilogue -- and a weight-gradient kernel (pixels are the reduction dimension: per-CTA register tiles of
//     16 x 32 (c_out x c_in*tap) accumulated over a grid-stride loop of 128-pixel chunks staged in shared memory,
//     per-CTA partials combined in a fixed order by one final kernel that can add  coef * gradient  straight into mu).
//
// Measured dead ends (kept out of the code): a 64-register weight-gradient kernel so that it co-resides with the data-gradient
// CTA (spills: 296 vs 287 us per adjoint stage); folding the producer warp into consumer warp 0 to fit two pipelined CTAs per SM
// at 128 registers (warp 0 stalls on the slowest warp every chunk: 147 vs 107 us per evaluation on block 2).
// The launch geometry (conv_grid, pipe_grid, cb_plan) is fixed at the measured best.
#include <math.h>

#include <map>

// The file is compiled twice, in parallel (pnode_b200/build.py): PNODE_CB_PART 1 = the fp32 instantiations + the C entry points,
// 2 = the fp64 instantiations.  0 (default, e.g. a plain `nvcc -c`) = everything in one object.
#ifndef PNODE_CB_PART
#define PNODE_CB_PART 0
#endif

#include "common.cuh"
#include "f32x2.cuh"
#include "pdl.cuh"

namespace pnode {

constexpr int CB_PGX = 64;   // pixel groups (4 pixels each) per CTA tile = blockDim.x
constexpr int CB_MAXCG = 4;  // channel groups per CTA = blockDim.y (<= 256 threads)
constexpr int ACC_R = 4;     // replicas of every accumulator (spreads the atomics of concurrently finishing CTAs)
enum { SRC_RAW = 0, SRC_ACT = 1, SRC_DZ = 2 };
enum { EPI_NONE = 0, EPI_FWD = 1, EPI_DGRAD = 2 };
#define FULL 0xffffffffu

template <typename T>
struct V4 {
    T v[4];
};

// acc += sum_e a[e] b[e] over four pixels (weight-gradient tiles)
template <typename T>
__device__ __forceinline__ void dot4_acc(const V4<T> &a, const V4<T> &b, T &acc) {
#pragma unroll
    for (int e = 0; e < 4; ++e) acc = fma(a.v[e], b.v[e], acc);
}

// acc[0..4) += w * o[0..4): four pixels of one output channel.  fp32: two packed FFMA2 (csrc/f32x2.cuh; the scalar weight is
// broadcast by the instruction, the pixel pairs are adjacent registers of the 128-bit load they came from) -- half the issue
// slots of four FFMA, identical rounding.
__device__ __forceinline__ void fma_row4(double w, const V4<double> &o, double (&acc)[4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[j] = fma(w, o.v[j], acc[j]);
}
__device__ __forceinline__ void fma_row4(float w, const V4<float> &o, float (&acc)[4]) {
    const F2 a = fma(w, pk(o.v[0], o.v[1]), pk(acc[0], acc[1]));
    const F2 b = fma(w, pk(o.v[2], o.v[3]), pk(acc[2], acc[3]));
    unpk(a, acc[0], acc[1]);
    unpk(b, acc[2], acc[3]);
}

__device__ __forceinline__ V4<float> ld4(const float *p) {
    const float4 t = *reinterpret_cast<const float4 *>(p);
    V4<float> r;
    r.v[0] = t.x, r.v[1] = t.y, r.v[2] = t.z, r.v[3] = t.w;
    return r;
}
__device__ __forceinline__ V4<double> ld4(const double *p) {
    const double2 a = *reinterpret_cast<const double2 *>(p), b = *reinterpret_cast<const double2 *>(p + 2);
    V4<double> r;
    r.v[0] = a.x, r.v[1] = a.y, r.v[2] = b.x, r.v[3] = b.y;
    return r;
}
__device__ __forceinline__ void st4(float *p, const V4<float> &r) {
    *reinterpret_cast<float4 *>(p) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
}
__device__ __forceinline__ void st4(double *p, const V4<double> &r) {
    *reinterpret_cast<double2 *>(p) = make_double2(r.v[0], r.v[1]);
    *reinterpret_cast<double2 *>(p + 2) = make_double2(r.v[2], r.v[3]);
}
template <typename T>
__device__ __forceinline__ V4<T> zero4() {
    V4<T> r;
    r.v[0] = r.v[1] = r.v[2] = r.v[3] = T(0);
    return r;
}

// ---- exact accumulators ---------------------------------------------------------------------------------------------------
// value = hi * 16 + lo * 2^-60 as a 128-bit two's-complement integer {lo: u64, hi: s64}; |x| < 2^66, resolution 8.7e-19.
// Adding is two integer atomics (the carry out of lo is known from the value the first atomic returns), so the total does
// not depend on the order of the adds.  Non-finite contributions raise *flag and the readers return NaN.
__device__ __forceinline__ void acc128_add(unsigned long long *p, double x, unsigned *flag) {
    if (!(fabs(x) < 7.0e19)) {
        atomicOr(flag, 1u);
        return;
    }
    const double m = fabs(x);
    const double h = floor(m * 0.0625);
    const double r = m - h * 16.0;  // exact (the low bits of m), in [0, 16)
    unsigned long long lo = (unsigned long long)(r * 1152921504606846976.0);  // 2^60; bits below 2^-60 are dropped
    long long hi = (long long)h;
    if (x < 0.0) {  // 128-bit two's-complement negation of the magnitude
        lo = ~lo + 1ull;
        hi = ~hi + (lo == 0ull ? 1 : 0);
    }
    const unsigned long long old = atomicAdd(p, lo);
    if (old + lo < old) hi += 1;
    if (hi != 0) atomicAdd(p + 1, (unsigned long long)hi);
}

// acc layout: [ACC_R][C][2 statistics][2 words]
__device__ __forceinline__ double acc128_read(const unsigned long long *acc, int C, int ch, int stat) {
    unsigned long long lo = 0;  // the replicas are added as 128-bit integers (exact); one conversion at the end
    long long hi = 0;
#pragma unroll
    for (int r = 0; r < ACC_R; ++r) {
        const unsigned long long *p = acc + (((int64_t)r * C + ch) * 2 + stat) * 2;
        const unsigned long long l = __ldcg(p);
        lo += l;
        hi += (long long)__ldcg(p + 1) + (lo < l ? 1 : 0);
    }
    const bool neg = hi < 0;  // convert the magnitude: a small negative total is hi = -1, lo = 2^64 - small
    if (neg) {
        lo = ~lo + 1ull;
        hi = ~hi + (lo == 0ull ? 1 : 0);
    }
    const double v = (double)hi * 16.0 + (double)lo * 8.673617379884035e-19;  // 2^-60
    return neg ? -v : v;
}

// One BatchNorm layer as the kernels see it: where its statistics accumulate and its affine parameters / buffers.
struct BnRef {
    const unsigned long long *accF;  // sum z, sum z^2                       (forward)
    const unsigned long long *accB;  // sum [y>0] g, sum [y>0] g xhat        (backward: dbeta, dgamma)
    const void *gamma, *beta;
    void *rmean, *rvar;
    long long *nbt;
    double eps, momentum;
    int C;
};

struct FwdStats {
    double mean, var, invstd, scale, shift;
};
template <typename T>
__device__ __forceinline__ FwdStats bn_forward_stats(const BnRef &b, int ch, double M, const unsigned *flag) {
    FwdStats f;
    const double bad = __ldcg(flag) != 0u ? NAN : 0.0;
    const double S = acc128_read(b.accF, b.C, ch, 0) + bad, Q = acc128_read(b.accF, b.C, ch, 1);
    f.mean = S / M;
    f.var = fmax(Q / M - f.mean * f.mean, 0.0);
    f.invstd = 1.0 / sqrt(f.var + b.eps);
    f.scale = (double)static_cast<const T *>(b.gamma)[ch] * f.invstd;
    f.shift = (double)static_cast<const T *>(b.beta)[ch] - f.mean * f.scale;
    return f;
}

// nn.BatchNorm2d's buffer update (momentum, unbiased variance), done once per evaluation by ONE CTA of the first consumer
template <typename T>
__device__ __forceinline__ void bn_update_running(const BnRef &b, double M, const unsigned *flag, int tid, int nthr) {
    if (b.rmean != nullptr) {
        T *rm = static_cast<T *>(b.rmean), *rv = static_cast<T *>(b.rvar);
        for (int ch = tid; ch < b.C; ch += nthr) {
            const FwdStats f = bn_forward_stats<T>(b, ch, M, flag);
            const double unbiased = M > 1.0 ? f.var * M / (M - 1.0) : f.var;
            rm[ch] = (T)((1.0 - b.momentum) * (double)rm[ch] + b.momentum * f.mean);
            rv[ch] = (T)((1.0 - b.momentum) * (double)rv[ch] + b.momentum * unbiased);
        }
    }
    if (tid == 0 && b.nbt != nullptr) *b.nbt += 1;
}

// per-channel coefficient tables in shared memory: [k][C], k-th coefficient of every channel
enum { CF_SCALE = 0, CF_SHIFT = 1, CF_MEAN = 2, CF_C0 = 3, CF_C1 = 4, CF_C2 = 5, CF_INVSTD = 3 };
template <int SRC>
struct NCoef {
    static constexpr int N = SRC == SRC_RAW ? 0 : (SRC == SRC_ACT ? 2 : 6);
};

// table of the INPUT-side coefficients of channels [c0, c0 + n): relu(bn(z)) = max(scale z + shift, 0) and, for SRC_DZ,
// dz = c0 [scale z + shift > 0] g + c1 (z - mean) + c2
template <typename T, int SRC>
__device__ __forceinline__ void fill_input_coefs(T *tab, int stride, const BnRef &b, int c0, int n, double M, const unsigned *flag,
                                                 int tid, int nthr) {
    if constexpr (SRC != SRC_RAW) {
        for (int i = tid; i < n; i += nthr) {
            const int ch = c0 + i;
            const FwdStats f = bn_forward_stats<T>(b, ch, M, flag);
            tab[CF_SCALE * stride + i] = (T)f.scale;
            tab[CF_SHIFT * stride + i] = (T)f.shift;
            if constexpr (SRC == SRC_DZ) {
                const double s1 = acc128_read(b.accB, b.C, ch, 0), s2 = acc128_read(b.accB, b.C, ch, 1);
                tab[CF_MEAN * stride + i] = (T)f.mean;
                tab[CF_C0 * stride + i] = (T)f.scale;
                tab[CF_C1 * stride + i] = (T)(-f.scale * f.invstd * s2 / M);
                tab[CF_C2 * stride + i] = (T)(-f.scale * s1 / M);
            }
        }
    }
}

// table of the OUTPUT-side coefficients (data-gradient epilogue): scale, shift, mean, inv-std of the layer below
template <typename T>
__device__ __forceinline__ void fill_output_coefs(T *tab, int stride, const BnRef &b, int c0, int n, double M, const unsigned *flag,
                                                  int tid, int nthr) {
    for (int i = tid; i < n; i += nthr) {
        const FwdStats f = bn_forward_stats<T>(b, c0 + i, M, flag);
        tab[CF_SCALE * stride + i] = (T)f.scale;
        tab[CF_SHIFT * stride + i] = (T)f.shift;
        tab[CF_MEAN * stride + i] = (T)f.mean;
        tab[CF_INVSTD * stride + i] = (T)f.invstd;
    }
}

// ---- what a kernel reads: the raw tensor, relu(bn(z)) formed on load, or the BatchNorm+ReLU backward formed on load -------
// Split into fetch(offset) / finish(channel, data) so that a kernel can issue the loads of several channels back to back
// (memory-level parallelism) before it starts consuming them.  `tab` is the shared-memory coefficient table.
template <typename T, int SRC>
struct Source;

template <typename T>
struct Source<T, SRC_RAW> {
    struct Data {
        V4<T> a;
    };
    const T *p;
    __device__ __forceinline__ Source(const T *a, const T *, const T *, int) : p(a) {}
    __device__ __forceinline__ Data fetch(int64_t off) const {
        Data d;
        d.a = ld4(p + off);
        return d;
    }
    __device__ __forceinline__ V4<T> finish(int, const Data &d) const { return d.a; }
};

template <typename T>
struct Source<T, SRC_ACT> {
    struct Data {
        V4<T> a;
    };
    const T *p, *tab;
    int stride;
    __device__ __forceinline__ Source(const T *a, const T *, const T *t, int s) : p(a), tab(t), stride(s) {}
    __device__ __forceinline__ Data fetch(int64_t off) const {
        Data d;
        d.a = ld4(p + off);
        return d;
    }
    __device__ __forceinline__ V4<T> finish(int i, const Data &d) const {
        const T sc = tab[CF_SCALE * stride + i], sh = tab[CF_SHIFT * stride + i];
        V4<T> v;
#pragma unroll
        for (int e = 0; e < 4; ++e) v.v[e] = fmax(fma(sc, d.a.v[e], sh), T(0));
        return v;
    }
};

template <typename T>
struct Source<T, SRC_DZ> {
    struct Data {
        V4<T> g, z;
    };
    const T *g, *z, *tab;
    int stride;
    __device__ __forceinline__ Source(const T *a, const T *b, const T *t, int s) : g(a), z(b), tab(t), stride(s) {}
    __device__ __forceinline__ Data fetch(int64_t off) const {
        Data d;
        d.g = ld4(g + off);
        d.z = ld4(z + off);
        return d;
    }
    __device__ __forceinline__ V4<T> finish(int i, const Data &d) const {
        const T sc = tab[CF_SCALE * stride + i], sh = tab[CF_SHIFT * stride + i], mean = tab[CF_MEAN * stride + i];
        const T c0 = tab[CF_C0 * stride + i], c1 = tab[CF_C1 * stride + i], c2 = tab[CF_C2 * stride + i];
        V4<T> r;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const T base = fma(c1, d.z.v[e] - mean, c2);
            r.v[e] = fma(sc, d.z.v[e], sh) > T(0) ? fma(c0, d.g.v[e], base) : base;
        }
        return r;
    }
};

// KIND 0: 1x1.  KIND 1: (1,3) pad (0,1): offsets -1, 0, +1 along W.  KIND 2: (3,1) pad (1,0): offsets -W, 0, +W.
// fetch_offsets issues the loads (KIND 2: the rows above / below, clamped at the image border so that every load is
// unconditional); finish_offsets turns them into o[i] = the 4 source values at offset (i - 1) of the thread's 4 pixels, zero
// outside the image.  finish_offsets must be called by all 32 lanes of a warp (KIND 1 shuffles); lanes hold consecutive pixel
// groups and a warp covers whole image rows.  Lanes past the end of the tensor read pixel group 0 and are never stored.
template <typename T, int KIND, typename S>
__device__ __forceinline__ void fetch_offsets(const S &src, int64_t off, int h, int H, int W,
                                              typename S::Data (&d)[KIND == 2 ? 3 : 1]) {
    if constexpr (KIND == 2) {
        d[0] = src.fetch(off - (h > 0 ? W : 0));
        d[1] = src.fetch(off);
        d[2] = src.fetch(off + (h < H - 1 ? W : 0));
    } else {
        d[0] = src.fetch(off);
    }
}

template <typename T, int KIND, typename S>
__device__ __forceinline__ void finish_offsets(const S &src, int i, const typename S::Data (&d)[KIND == 2 ? 3 : 1], int h, int w0,
                                               int H, int W, V4<T> (&o)[KIND == 0 ? 1 : 3]) {
    if constexpr (KIND == 0) {
        o[0] = src.finish(i, d[0]);
    } else if constexpr (KIND == 1) {
        const V4<T> c = src.finish(i, d[0]);
        T l = __shfl_up_sync(FULL, c.v[3], 1), r = __shfl_down_sync(FULL, c.v[0], 1);
        if (w0 == 0) l = T(0);
        if (w0 + 4 == W) r = T(0);
        o[0].v[0] = l, o[0].v[1] = c.v[0], o[0].v[2] = c.v[1], o[0].v[3] = c.v[2];
        o[1] = c;
        o[2].v[0] = c.v[1], o[2].v[1] = c.v[2], o[2].v[2] = c.v[3], o[2].v[3] = r;
    } else {
        o[0] = h > 0 ? src.finish(i, d[0]) : zero4<T>();
        o[1] = src.finish(i, d[1]);
        o[2] = h < H - 1 ? src.finish(i, d[2]) : zero4<T>();
    }
}

// input channels per register buffer (two buffers are live: the group being consumed and the group in flight)
template <int KIND, int SRC>
struct Unroll {
    static constexpr int N = KIND == 2 ? (SRC == SRC_DZ ? 1 : 2) : (SRC == SRC_DZ ? 2 : 4);
};

struct PixelCoord {
    int n, rem, h, w0;
    bool active;
};
__device__ __forceinline__ PixelCoord pixel_coord(int64_t pg, int64_t npg, int HW, int W) {
    PixelCoord c;
    c.active = pg < npg;
    const int64_t q = c.active ? pg * 4 : 0;
    c.n = (int)(q / HW);
    c.rem = (int)(q - (int64_t)c.n * HW);
    c.h = c.rem / W;
    c.w0 = c.rem - c.h * W;
    return c;
}

template <typename T>
struct ConvArgs {
    const T *in, *in2;   // forward: z_{k-1} (or x), unused;  data gradient: g_k, z_k
    const T *w, *bias;   // conv weight [Cout][Cin][taps]; bias [Cout] (forward only)
    T *out;              // forward: z_k;  data gradient: g_{k-1} (or the VJP w.r.t. the block input)
    const T *zprev;      // EPI_DGRAD: z_{k-1} at the output pixels
    BnRef bin, bout;     // BatchNorm on the input side (forward: layer k-1; dgrad: layer k) / output side (dgrad: layer k-1)
    unsigned long long *acc_out;  // accumulators this kernel adds into (forward: accF of layer k; dgrad: accB of layer k-1)
    unsigned *flag;
    unsigned *ticket;                      // data-parallel runs: CTA completion counter of the kernel (self-resetting)
    const unsigned long long *peer_bufs;   // DEVICE array [world]: peer-mapped base of every rank's symmetric inbox, or NULL
    unsigned long long epoch;              // collective number of this kernel's statistics exchange (consecutive, all ranks)
    int rank, world;
    int upd_in, upd_out;  // CTA (0,0) performs the running-statistics update of bin / bout
    int CA, CB;           // reduction channels, output channels
    int H, W, HW;
    int64_t npg;          // pixel groups = N*H*W/4
    int tiles;
    double M;             // N*H*W
};

// 2*RC per-thread values summed over the 32 lanes with a transposing butterfly (2*RC + log-ish shuffles instead of 5 per
// value): on return lane l holds the warp total of value index idx(l) (the top log2(NV) bits of l, MSB first).
template <typename T, int NV>
__device__ __forceinline__ T warp_multi_sum(T (&v)[NV], int lane, int &idx) {
    idx = 0;
    int bit = 16;
#pragma unroll
    for (int n = NV / 2; n >= 1; n >>= 1, bit >>= 1) {
        const bool hi = (lane & bit) != 0;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            const T send = hi ? v[i] : v[i + n];
            const T keep = hi ? v[i + n] : v[i];
            v[i] = keep + __shfl_xor_sync(FULL, send, bit);
        }
        idx = idx * 2 + (hi ? 1 : 0);
    }
    T t = v[0];
    for (; bit >= 1; bit >>= 1) t += __shfl_xor_sync(FULL, t, bit);
    return t;
}

template <bool NAMED>
__device__ __forceinline__ void cta_sync() {
    if constexpr (NAMED) asm volatile("bar.sync 1, 256;" ::: "memory");
    else __syncthreads();
}

// Batch-sharded runs (one process per GPU): the batch statistics must be those of the GLOBAL batch.  Compute and collective in
// one kernel: the last CTA of this rank (ticket) folds the accumulator replicas into exact 128-bit totals, stores them into
// every rank's symmetric-memory inbox over NVLink (plain st.global on peer-mapped addresses), raises a system-scope release
// flag, waits for the other ranks' flags, sums the inbox -- integer sums: every rank gets the same bits whatever the order --
// and writes the global totals back as THE accumulator, so every consumer (next kernel, saved activation sets, the adjoint)
// is unchanged.  Same inbox / flag / epoch protocol as common.cuh:peer_allreduce_and_store (two sets alternate by epoch).
template <typename T, bool NAMED>
__device__ __forceinline__ void stats_exchange(const ConvArgs<T> &a, int tid, int nthr) {
    if (a.world <= 1 || a.peer_bufs == nullptr) return;
    __shared__ int is_last;
    __threadfence();
    cta_sync<NAMED>();
    if (tid == 0) is_last = atomicAdd(a.ticket, 1u) == gridDim.x * gridDim.y - 1;
    cta_sync<NAMED>();
    if (!is_last) return;
    __threadfence();
    const int nval = 2 * a.CB, set = (int)(a.epoch & 1ull);
    for (int v = tid; v < nval; v += nthr) {
        unsigned long long lo = 0;
        long long hi = 0;
        for (int r = 0; r < ACC_R; ++r) {
            const unsigned long long *p = a.acc_out + ((int64_t)r * nval + v) * 2;
            const unsigned long long l = __ldcg(p);
            lo += l;
            hi += (long long)__ldcg(p + 1) + (lo < l ? 1 : 0);
        }
        for (int r = 0; r < a.world; ++r) {
            unsigned long long *dst = reinterpret_cast<unsigned long long *>(peer_slot(a.peer_bufs[r], set, a.world, a.rank));
            dst[2 * v] = lo;
            dst[2 * v + 1] = (unsigned long long)hi;
        }
    }
    __threadfence_system();
    cta_sync<NAMED>();
    if (tid < a.world) {
        unsigned long long *f = peer_flag(a.peer_bufs[tid], set, a.world, a.rank);
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(f), "l"(a.epoch) : "memory");
        unsigned long long *w = peer_flag(a.peer_bufs[a.rank], set, a.world, tid), v = 0;
        for (long long spin = 0; spin < (1ll << 27); ++spin) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(w) : "memory");
            if (v >= a.epoch) break;
            __nanosleep(64);
        }
        if (v < a.epoch) atomicOr(a.flag, 2u);  // a peer never arrived: poison the statistics instead of hanging
    }
    cta_sync<NAMED>();
    const unsigned long long mine = a.peer_bufs[a.rank];
    for (int v = tid; v < nval; v += nthr) {
        unsigned long long lo = 0;
        long long hi = 0;
        for (int r = 0; r < a.world; ++r) {
            const unsigned long long *src = reinterpret_cast<const unsigned long long *>(peer_slot(mine, set, a.world, r));
            const unsigned long long l = __ldcg(src + 2 * v);
            lo += l;
            hi += (long long)__ldcg(src + 2 * v + 1) + (lo < l ? 1 : 0);
        }
        a.acc_out[2 * v] = lo;
        a.acc_out[2 * v + 1] = (unsigned long long)hi;
        for (int r = 1; r < ACC_R; ++r) a.acc_out[((int64_t)r * nval + v) * 2] = 0ull, a.acc_out[((int64_t)r * nval + v) * 2 + 1] = 0ull;
    }
    if (tid == 0) *a.ticket = 0u;
}

// CTA-level sums of the per-thread statistics, added into the exact accumulators (no tail, no ordering)
template <typename T, int RC>
__device__ __forceinline__ void stats_epilogue(const ConvArgs<T> &a, T (&s)[RC], T (&q)[RC], int cb0) {
    __shared__ double red[2][CB_MAXCG][2 * RC];
    const int lane = threadIdx.x & 31, wx = threadIdx.x >> 5;
    T v[2 * RC];
#pragma unroll
    for (int r = 0; r < RC; ++r) v[r] = s[r], v[RC + r] = q[r];
    int idx;
    const T t = warp_multi_sum<T, 2 * RC>(v, lane, idx);
    constexpr int REP = 32 / (2 * RC);  // lanes sharing idx hold the same total; one of them publishes it
    if ((lane & (REP - 1)) == 0) red[wx][threadIdx.y][idx] = (double)t;
    __syncthreads();
    if (threadIdx.x < 2 * RC) {
        const int which = threadIdx.x / RC, r = threadIdx.x % RC;
        const int ch = cb0 + threadIdx.y * RC + r;
        const int rep = blockIdx.x % ACC_R;
        acc128_add(a.acc_out + (((int64_t)rep * a.CB + ch) * 2 + which) * 2,
                   red[0][threadIdx.y][threadIdx.x] + red[1][threadIdx.y][threadIdx.x], a.flag);
    }
    stats_exchange<T, false>(a, threadIdx.y * CB_PGX + threadIdx.x, CB_PGX * blockDim.y);
}

// sum / sum-of-squares (forward) or the two BatchNorm-backward sums (dgrad) of one thread's RC x 4 outputs
template <typename T, int RC, int EPI>
__device__ __forceinline__ void stats_accumulate(const ConvArgs<T> &a, const T (&acc)[RC][4], int64_t off_out, const T *tout,
                                                 int tstride, int i0, T (&s)[RC], T (&q)[RC]) {
    if constexpr (EPI == EPI_FWD) {
#pragma unroll
        for (int r = 0; r < RC; ++r)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                s[r] += acc[r][j];
                q[r] = fma(acc[r][j], acc[r][j], q[r]);
            }
    } else {
        V4<T> z[RC];
#pragma unroll
        for (int r = 0; r < RC; ++r) z[r] = ld4(a.zprev + off_out + (int64_t)r * a.HW);
#pragma unroll
        for (int r = 0; r < RC; ++r) {
            const T sc = tout[CF_SCALE * tstride + i0 + r], sh = tout[CF_SHIFT * tstride + i0 + r];
            const T mean = tout[CF_MEAN * tstride + i0 + r], invstd = tout[CF_INVSTD * tstride + i0 + r];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const T gm = fma(sc, z[r].v[j], sh) > T(0) ? acc[r][j] : T(0);
                s[r] += gm;
                q[r] = fma(gm, (z[r].v[j] - mean) * invstd, q[r]);
            }
        }
    }
}

template <typename T>
__device__ __forceinline__ V4<T> lds4(const T *p) {
    return ld4(p);
}

// out[b][pixel] = bias[b] + sum_{a, offset} Wsel[a][offset][b] * src(a, pixel + offset)
template <typename T, int KIND, int SRC, int EPI, int RC>
__global__ void __launch_bounds__(CB_PGX *CB_MAXCG) conv_kernel(const ConvArgs<T> a) {
    constexpr int TAPS = KIND == 0 ? 1 : 3;
    constexpr bool FWD = SRC != SRC_DZ;
    constexpr int UN = Unroll<KIND, SRC>::N, NF = KIND == 2 ? 3 : 1;
    typedef Source<T, SRC> S;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int CT = blockDim.y * RC;
    T *ws = reinterpret_cast<T *>(smem_raw);  // [CA * TAPS][CT]
    T *tin = ws + a.CA * TAPS * CT;           // [NCoef][CA]
    T *tout = tin + NCoef<SRC>::N * a.CA;     // [4][CT]   (EPI_DGRAD)
    const int cb0 = blockIdx.y * CT;
    const int tid = threadIdx.y * CB_PGX + threadIdx.x, nthr = CB_PGX * blockDim.y;
    pdl::pdl_launch_dependents();
    for (int i = tid; i < a.CA * TAPS * CT; i += nthr) {
        const int bl = i % CT, ao = i / CT, o = ao % TAPS, ach = ao / TAPS, b = cb0 + bl;
        // forward: W[co = b][ci = ach][tap = o];  data gradient: W[co = ach][ci = b][tap = TAPS-1-o]
        ws[i] = FWD ? a.w[((int64_t)b * a.CA + ach) * TAPS + o] : a.w[((int64_t)ach * a.CB + b) * TAPS + (TAPS - 1 - o)];
    }
    pdl::pdl_wait();
    fill_input_coefs<T, SRC>(tin, a.CA, a.bin, 0, a.CA, a.M, a.flag, tid, nthr);
    if constexpr (EPI == EPI_DGRAD) fill_output_coefs<T>(tout, CT, a.bout, cb0, CT, a.M, a.flag, tid, nthr);
    if (blockIdx.x == 0 && blockIdx.y == 0) {
        if (a.upd_in) bn_update_running<T>(a.bin, a.M, a.flag, tid, nthr);
        if (a.upd_out) bn_update_running<T>(a.bout, a.M, a.flag, tid, nthr);
    }
    __syncthreads();
    S src(a.in, a.in2, tin, a.CA);
    const int ch0 = cb0 + threadIdx.y * RC;
    T bias[RC], s[RC], q[RC];
#pragma unroll
    for (int r = 0; r < RC; ++r) {
        bias[r] = (FWD && a.bias != nullptr) ? a.bias[ch0 + r] : T(0);
        s[r] = q[r] = T(0);
    }
    for (int tile = blockIdx.x; tile < a.tiles; tile += gridDim.x) {
        const PixelCoord pc = pixel_coord((int64_t)tile * CB_PGX + threadIdx.x, a.npg, a.HW, a.W);
        const int64_t off_in = (int64_t)pc.n * a.CA * a.HW + pc.rem;
        T acc[RC][4];
#pragma unroll
        for (int r = 0; r < RC; ++r)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[r][j] = bias[r];
        typename S::Data cur[UN][NF], nxt[UN][NF];
#pragma unroll
        for (int u = 0; u < UN; ++u) fetch_offsets<T, KIND>(src, off_in + (int64_t)u * a.HW, pc.h, a.H, a.W, cur[u]);
        for (int cb = 0; cb < a.CA; cb += UN) {  // host guarantees CA % 4 == 0
            const bool more = cb + UN < a.CA;
            if (more) {
#pragma unroll
                for (int u = 0; u < UN; ++u)
                    fetch_offsets<T, KIND>(src, off_in + (int64_t)(cb + UN + u) * a.HW, pc.h, a.H, a.W, nxt[u]);
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                V4<T> o[TAPS];
                finish_offsets<T, KIND>(src, cb + u, cur[u], pc.h, pc.w0, a.H, a.W, o);
#pragma unroll
                for (int oi = 0; oi < TAPS; ++oi) {
                    const T *wr = ws + ((cb + u) * TAPS + oi) * CT + threadIdx.y * RC;
#pragma unroll
                    for (int r4 = 0; r4 < RC; r4 += 4) {
                        const V4<T> wv = lds4<T>(wr + r4);
#pragma unroll
                        for (int r = 0; r < 4; ++r) fma_row4(wv.v[r], o[oi], acc[r4 + r]);
                    }
                }
            }
            if (more) {
#pragma unroll
                for (int u = 0; u < UN; ++u)
#pragma unroll
                    for (int f = 0; f < NF; ++f) cur[u][f] = nxt[u][f];
            }
        }
        if (pc.active) {
            const int64_t off_out = ((int64_t)pc.n * a.CB + ch0) * a.HW + pc.rem;
#pragma unroll
            for (int r = 0; r < RC; ++r) {
                V4<T> v;
#pragma unroll
                for (int j = 0; j < 4; ++j) v.v[j] = acc[r][j];
                st4(a.out + off_out + (int64_t)r * a.HW, v);
            }
            if constexpr (EPI != EPI_NONE) stats_accumulate<T, RC, EPI>(a, acc, off_out, tout, CT, threadIdx.y * RC, s, q);
        }
    }
    if constexpr (EPI != EPI_NONE) stats_epilogue<T, RC>(a, s, q, cb0);
}

// ---- pipelined variant: TMA bulk copies (cp.async.bulk, no tensor map: a tile of one channel of one image is contiguous in
// NCHW) feed a ring of shared-memory stages through mbarriers; one producer warp, eight consumer warps --------------------
// CTA tile = TP = 1024 / CG consecutive pixels (whole images when HW <= TP, else a row range of one image) x CT = CG * RC
// output channels; a stage holds KC input channels of the tile, raw (the BatchNorm+ReLU / backward transform is applied when
// a consumer reads its 4 pixels out of shared memory, so each activation is transformed once per channel group).  The copies
// of up to S stages are in flight while the consumers run FMAs, across tile boundaries too: the grid is persistent.
constexpr int CP_CONSUMERS = 256;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok = 0;
    for (long long spin = 0; spin < (1ll << 26); ++spin) {  // bounded: a protocol bug must not hang the GPU
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (ok) return;
    }
    __trap();
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

template <int SRC>
struct PipeKC {
    static constexpr int N = SRC == SRC_DZ ? 2 : 4;  // input channels per stage (SRC_DZ stages two tensors)
};

template <typename T, int KIND, int SRC, int EPI, int RC>
__global__ void __launch_bounds__(CP_CONSUMERS + 32) convp_kernel(const ConvArgs<T> a, const int CG, const int S) {
    constexpr int TAPS = KIND == 0 ? 1 : 3;
    constexpr bool FWD = SRC != SRC_DZ;
    constexpr int KC = PipeKC<SRC>::N, NT = SRC == SRC_DZ ? 2 : 1, NF = KIND == 2 ? 3 : 1;
    typedef Source<T, SRC> SS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int CT = CG * RC, PGT = CP_CONSUMERS / CG, TP = 4 * PGT;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem_raw), *empty = full + 8;
    T *ws = reinterpret_cast<T *>(smem_raw + 128);  // [CA * TAPS][CT]
    T *tin = ws + a.CA * TAPS * CT;                 // [NCoef][CA]
    T *tout = tin + NCoef<SRC>::N * a.CA;           // [4][CT]
    const size_t head = (128 + ((size_t)a.CA * TAPS * CT + (size_t)NCoef<SRC>::N * a.CA + 4 * CT) * sizeof(T) + 127) & ~(size_t)127;
    T *stages = reinterpret_cast<T *>(smem_raw + head);  // [S][NT][KC][TP]
    const int stage_elems = NT * KC * TP;
    const int cb0 = blockIdx.y * CT;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nchunk = a.CA / KC;
    const int ipt = TP >= a.HW ? TP / a.HW : 0;  // images per tile (0: the tile is a row range of one image)
    const int64_t total_px = a.npg * 4;
    if (tid == 0) {
        for (int i = 0; i < S; ++i) {
            mbar_init(full + i, 1);
            mbar_init(empty + i, CP_CONSUMERS / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    pdl::pdl_launch_dependents();
    __syncthreads();
    if (warp == CP_CONSUMERS / 32) {
        pdl::pdl_wait();
        // ---- producer warp: every lane issues a share of the stage's bulk copies; lane 0 arms the barrier -------------------
        int slot = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < a.tiles; tile += gridDim.x) {
            const int64_t px0 = (int64_t)tile * TP;
            int imgs, n0, rem0;
            uint32_t bytes_each;
            if (ipt > 0) {
                n0 = tile * ipt, rem0 = 0;
                const int64_t left = (total_px - px0) / a.HW;
                imgs = (int)(left < ipt ? left : ipt);
                bytes_each = (uint32_t)(a.HW * sizeof(T));
            } else {
                n0 = (int)(px0 / a.HW), rem0 = (int)(px0 - (int64_t)n0 * a.HW);
                imgs = 1;
                bytes_each = (uint32_t)(TP * sizeof(T));
            }
            const int ncopy = NT * KC * imgs;
            for (int chunk = 0; chunk < nchunk; ++chunk) {
                mbar_wait(empty + slot, phase ^ 1u);
                T *st = stages + (size_t)slot * stage_elems;
                if (lane == 0) mbar_expect_tx(full + slot, bytes_each * (uint32_t)ncopy);
                __syncwarp();
                for (int i = lane; i < ncopy; i += 32) {
                    const int m = i % imgs, tc = i / imgs, c = tc % KC, t = tc / KC;
                    const T *base = (t == 0) ? a.in : a.in2;
                    const T *src = base + ((int64_t)(n0 + m) * a.CA + chunk * KC + c) * a.HW + rem0;
                    bulk_g2s(st + (t * KC + c) * TP + m * a.HW, src, bytes_each, full + slot);
                }
                if (++slot == S) slot = 0, phase ^= 1u;
            }
        }
        return;
    }
    // ---- consumers ------------------------------------------------------------------------------------------------------------
    const int x = tid % PGT, cg = tid / PGT;
    for (int i = tid; i < a.CA * TAPS * CT; i += CP_CONSUMERS) {
        const int bl = i % CT, ao = i / CT, o = ao % TAPS, ach = ao / TAPS, b = cb0 + bl;
        ws[i] = FWD ? a.w[((int64_t)b * a.CA + ach) * TAPS + o] : a.w[((int64_t)ach * a.CB + b) * TAPS + (TAPS - 1 - o)];
    }
    pdl::pdl_wait();
    fill_input_coefs<T, SRC>(tin, a.CA, a.bin, 0, a.CA, a.M, a.flag, tid, CP_CONSUMERS);
    if constexpr (EPI == EPI_DGRAD) fill_output_coefs<T>(tout, CT, a.bout, cb0, CT, a.M, a.flag, tid, CP_CONSUMERS);
    if (blockIdx.x == 0 && blockIdx.y == 0) {
        if (a.upd_in) bn_update_running<T>(a.bin, a.M, a.flag, tid, CP_CONSUMERS);
        if (a.upd_out) bn_update_running<T>(a.bout, a.M, a.flag, tid, CP_CONSUMERS);
    }
    consumer_sync();
    const int ch0 = cb0 + cg * RC;
    __shared__ double red[CP_CONSUMERS / 32][2 * RC];
    int slot = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < a.tiles; tile += gridDim.x) {
        const PixelCoord pc = pixel_coord((int64_t)tile * PGT + x, a.npg, a.HW, a.W);
        const int xo = pc.active ? 4 * x : 0;  // lanes past the end of the tensor read the tile's first pixels (never stored)
        T acc[RC][4];
#pragma unroll
        for (int r = 0; r < RC; ++r) {
            const T b = (FWD && a.bias != nullptr) ? __ldg(a.bias + ch0 + r) : T(0);
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[r][j] = b;
        }
        for (int chunk = 0; chunk < nchunk; ++chunk) {
            mbar_wait(full + slot, phase);
            const T *st = stages + (size_t)slot * stage_elems;
            SS src(st, st + KC * TP, tin, a.CA);
            typename SS::Data dd[KC][NF];
#pragma unroll
            for (int c = 0; c < KC; ++c) fetch_offsets<T, KIND>(src, (int64_t)c * TP + xo, pc.h, a.H, a.W, dd[c]);
#pragma unroll
            for (int c = 0; c < KC; ++c) {
                const int ch = chunk * KC + c;
                V4<T> o[TAPS];
                finish_offsets<T, KIND>(src, ch, dd[c], pc.h, pc.w0, a.H, a.W, o);
#pragma unroll
                for (int oi = 0; oi < TAPS; ++oi) {
                    const T *wr = ws + (ch * TAPS + oi) * CT + cg * RC;
#pragma unroll
                    for (int r4 = 0; r4 < RC; r4 += 4) {
                        const V4<T> wv = lds4<T>(wr + r4);
#pragma unroll
                        for (int r = 0; r < 4; ++r) fma_row4(wv.v[r], o[oi], acc[r4 + r]);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(empty + slot);
            if (++slot == S) slot = 0, phase ^= 1u;
        }
        // per-TILE statistics (not carried across tiles in registers: the main loop keeps its registers, and a tile's partial
        // sums do not depend on how tiles are spread over CTAs)
        T s[RC], q[RC];
#pragma unroll
        for (int r = 0; r < RC; ++r) s[r] = q[r] = T(0);
        if (pc.active) {
            const int64_t off_out = ((int64_t)pc.n * a.CB + ch0) * a.HW + pc.rem;
#pragma unroll
            for (int r = 0; r < RC; ++r) {
                V4<T> v;
#pragma unroll
                for (int j = 0; j < 4; ++j) v.v[j] = acc[r][j];
                st4(a.out + off_out + (int64_t)r * a.HW, v);
            }
            if constexpr (EPI != EPI_NONE) stats_accumulate<T, RC, EPI>(a, acc, off_out, tout, CT, cg * RC, s, q);
        }
        if constexpr (EPI != EPI_NONE) {
            T v[2 * RC];
#pragma unroll
            for (int r = 0; r < RC; ++r) v[r] = s[r], v[RC + r] = q[r];
            int idx;
            const T t = warp_multi_sum<T, 2 * RC>(v, lane, idx);
            constexpr int REP = 32 / (2 * RC);
            if ((lane & (REP - 1)) == 0) red[warp][idx] = (double)t;
            consumer_sync();
            if (tid < 2 * CT) {
                const int g = tid / (2 * RC), i = tid % (2 * RC), which = i / RC, r = i % RC;
                const int wpg = PGT / 32;  // warps per channel group
                double tot = 0.0;
                for (int w = 0; w < wpg; ++w) tot += red[g * wpg + w][i];
                const int ch = cb0 + g * RC + r;
                const int rep = tile % ACC_R;
                acc128_add(a.acc_out + (((int64_t)rep * a.CB + ch) * 2 + which) * 2, tot, a.flag);
            }
            consumer_sync();
        }
    }
    if constexpr (EPI != EPI_NONE) stats_exchange<T, true>(a, tid, CP_CONSUMERS);
}

// BatchNorm-backward sums of the TOP layer (g = the cotangent handed to the VJP, z = z_L): same epilogue, no convolution.
template <typename T, int RC>
__global__ void __launch_bounds__(CB_PGX *CB_MAXCG) top_stats_kernel(const ConvArgs<T> a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T *tout = reinterpret_cast<T *>(smem_raw);  // [4][CT]
    const int CT = blockDim.y * RC;
    const int cb0 = blockIdx.y * CT, ch0 = cb0 + threadIdx.y * RC;
    const int tid = threadIdx.y * CB_PGX + threadIdx.x, nthr = CB_PGX * blockDim.y;
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    fill_output_coefs<T>(tout, CT, a.bout, cb0, CT, a.M, a.flag, tid, nthr);
    if (blockIdx.x == 0 && blockIdx.y == 0 && a.upd_out) bn_update_running<T>(a.bout, a.M, a.flag, tid, nthr);
    __syncthreads();
    T s[RC], q[RC];
#pragma unroll
    for (int r = 0; r < RC; ++r) s[r] = q[r] = T(0);
    for (int tile = blockIdx.x; tile < a.tiles; tile += gridDim.x) {
        const PixelCoord pc = pixel_coord((int64_t)tile * CB_PGX + threadIdx.x, a.npg, a.HW, a.W);
        if (!pc.active) continue;
        const int64_t off_out = ((int64_t)pc.n * a.CB + ch0) * a.HW + pc.rem;
        T acc[RC][4];
        V4<T> g[RC];
#pragma unroll
        for (int r = 0; r < RC; ++r) g[r] = ld4(a.in + off_out + (int64_t)r * a.HW);
#pragma unroll
        for (int r = 0; r < RC; ++r)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[r][j] = g[r].v[j];
        stats_accumulate<T, RC, EPI_DGRAD>(a, acc, off_out, tout, CT, threadIdx.y * RC, s, q);
    }
    stats_epilogue<T, RC>(a, s, q, cb0);
}

// out = base_coef * base + coef * relu(scale_c * z + shift_c)      (base may be NULL: plain activation of the last layer;
// with base it is the RK stage combination Y_{i+1} = u + h a_{i+1,i} k_i fused into the block's output pass)
template <typename T>
__global__ void __launch_bounds__(256) act_out_kernel(const T *__restrict__ z, const BnRef b, double M, const unsigned *flag,
                                                      int upd, int HW, int64_t nvec, T *__restrict__ out,
                                                      const T *__restrict__ base, T base_coef, T kcoef, T *__restrict__ kout) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T *tab = reinterpret_cast<T *>(smem_raw);  // [2][C]
    const int C = b.C;
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    fill_input_coefs<T, SRC_ACT>(tab, C, b, 0, C, M, flag, threadIdx.x, blockDim.x);
    if (blockIdx.x == 0 && upd) bn_update_running<T>(b, M, flag, threadIdx.x, blockDim.x);
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        const int64_t e0 = i * 4;
        const int c = (int)((e0 / HW) % C);
        const T sc = tab[CF_SCALE * C + c], sh = tab[CF_SHIFT * C + c];
        V4<T> v = ld4(z + e0);
#pragma unroll
        for (int e = 0; e < 4; ++e) v.v[e] = fmax(fma(sc, v.v[e], sh), T(0));
        if (kout != nullptr) st4(kout + e0, v);
        if (base != nullptr) {
            const V4<T> bb = ld4(base + e0);
#pragma unroll
            for (int e = 0; e < 4; ++e) v.v[e] = fma(kcoef, v.v[e], base_coef * bb.v[e]);
        }
        if (out != nullptr) st4(out + e0, v);
    }
}

// ---- weight gradient ------------------------------------------------------------------------------------------------------
// dW[co][ci][tap] = sum_pixels dz[co][p] * y[ci][p + tap - 1]: pixels are the reduction dimension.  A CTA owns one
// (4 TM) x (8 TN) tile of the (c_out) x (c_in * taps) gradient and a grid-stride share of the 128-pixel chunks; a chunk's dz
// rows and (tap-shifted) y rows are formed on load, staged pixel-major in shared memory, and every warp accumulates the tile
// over its own 16 pixels of the chunk (lane = 4 c_out groups x 8 c_in*tap groups, TM x TN register tile, LDS.128 along the
// pixels).  (TM, TN) is picked per layer so that the tile fits the layer's channel counts (block 1: 16x32, 8x16, 16x24,
// 16x48, 32x16).  The gradient of a convolution bias that feeds a BatchNorm is exactly zero (sum_p dz = 0) and is not computed.
constexpr int WG_PX = 128, WG_LD = 132, WG_THREADS = 256;

template <typename T>
struct WgradArgs {
    const T *g, *z;   // dz_k formed on load from g_k, z_k and layer k's statistics
    const T *yin;     // y_{k-1}: raw block input (k = 1) or relu(bn(z_{k-1}))
    BnRef bk, bin;    // layer k (forward + backward sums), layer k-1 (forward sums)
    const unsigned *flag;
    T *partial;       // [gridDim.x][gridDim.y][WG_CO * WG_CIT]
    int Cin, Cout, H, W, HW, tiles_cit;
    int64_t npg;
    int nchunks;
    double M;
};

template <typename T, int KIND, int YSRC, int TM, int TN>
__global__ void __launch_bounds__(WG_THREADS) conv_wgrad_kernel(const WgradArgs<T> a) {
    constexpr int TAPS = KIND == 0 ? 1 : 3;
    constexpr int WG_CO = 4 * TM, WG_CIT = 8 * TN, WG_TILE = WG_CO * WG_CIT;
    constexpr int NDZ = (WG_CO + 7) / 8;                                          // dz rows per warp
    constexpr int NY = TAPS == 1 ? (WG_CIT + 7) / 8 : (WG_CIT / 3 + 2 + 7) / 8;   // source channels per warp
    constexpr int NF = KIND == 2 ? 3 : 1;
    typedef Source<T, SRC_DZ> SD;
    typedef Source<T, YSRC> SY;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T *s_dz = reinterpret_cast<T *>(smem_raw);  // [WG_CO][WG_LD]
    T *s_y = s_dz + WG_CO * WG_LD;              // [WG_CIT][WG_LD]
    T *tdz = s_y + WG_CIT * WG_LD;              // [6][WG_CO]
    T *ty = tdz + 6 * WG_CO;                    // [2][WG_CIT]
    const int tile = blockIdx.y, tco = tile / a.tiles_cit, tcit = tile % a.tiles_cit;
    const int co0 = tco * WG_CO, cit0 = tcit * WG_CIT;
    const int ci_lo = cit0 / TAPS, ci_hi = min(a.Cin, (cit0 + WG_CIT - 1) / TAPS + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cgp = lane & 3, cg8 = lane >> 2;
    pdl::pdl_launch_dependents();
    for (int i = threadIdx.x; i < (WG_CO + WG_CIT) * WG_LD; i += WG_THREADS) s_dz[i] = T(0);
    pdl::pdl_wait();
    fill_input_coefs<T, SRC_DZ>(tdz, WG_CO, a.bk, co0, min(WG_CO, a.Cout - co0), a.M, a.flag, threadIdx.x, WG_THREADS);
    fill_input_coefs<T, YSRC>(ty, WG_CIT, a.bin, ci_lo, ci_hi - ci_lo, a.M, a.flag, threadIdx.x, WG_THREADS);
    __syncthreads();
    SD dsrc(a.g, a.z, tdz, WG_CO);
    SY ysrc(a.yin, nullptr, ty, WG_CIT);
    T acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = T(0);
    // this warp's rows of a chunk: NDZ dz rows (channels co0 + warp + 8 i) and NY source channels (ci_lo + warp + 8 u), clamped
    int rdz[NDZ], rci[NY];
#pragma unroll
    for (int i = 0; i < NDZ; ++i) rdz[i] = min(warp + 8 * i, min(WG_CO, a.Cout - co0) - 1);
#pragma unroll
    for (int u = 0; u < NY; ++u) rci[u] = min(warp + 8 * u, ci_hi - ci_lo - 1);
    typename SD::Data ddz[NDZ];
    typename SY::Data dy[NY][NF];
    PixelCoord pc = pixel_coord((int64_t)blockIdx.x * 32 + lane, a.npg, a.HW, a.W);
    auto fetch = [&](const PixelCoord &c) {
#pragma unroll
        for (int i = 0; i < NDZ; ++i) ddz[i] = dsrc.fetch(((int64_t)c.n * a.Cout + co0 + rdz[i]) * a.HW + c.rem);
#pragma unroll
        for (int u = 0; u < NY; ++u)
            fetch_offsets<T, KIND>(ysrc, ((int64_t)c.n * a.Cin + ci_lo + rci[u]) * a.HW + c.rem, c.h, a.H, a.W, dy[u]);
    };
    if ((int)blockIdx.x < a.nchunks) fetch(pc);
    for (int chunk = blockIdx.x; chunk < a.nchunks; chunk += gridDim.x) {
#pragma unroll
        for (int i = 0; i < NDZ; ++i) {
            const int r = warp + 8 * i;
            if (r < WG_CO && co0 + r < a.Cout)
                st4(s_dz + r * WG_LD + lane * 4, pc.active ? dsrc.finish(rdz[i], ddz[i]) : zero4<T>());
        }
#pragma unroll
        for (int u = 0; u < NY; ++u) {
            const int ci = ci_lo + warp + 8 * u;  // warp-uniform
            V4<T> o[TAPS];
            finish_offsets<T, KIND>(ysrc, rci[u], dy[u], pc.h, pc.w0, a.H, a.W, o);
            if (ci < ci_hi) {
#pragma unroll
                for (int oi = 0; oi < TAPS; ++oi) {
                    const int r = ci * TAPS + oi - cit0;
                    if (r >= 0 && r < WG_CIT) st4(s_y + r * WG_LD + lane * 4, pc.active ? o[oi] : zero4<T>());
                }
            }
        }
        __syncthreads();
        // the next chunk's loads fly while this one is consumed
        const int next = chunk + gridDim.x;
        if (next < a.nchunks) {
            pc = pixel_coord((int64_t)next * 32 + lane, a.npg, a.HW, a.W);
            fetch(pc);
        }
#pragma unroll
        for (int pp = 0; pp < WG_PX / 8; pp += 4) {
            const int p = warp * (WG_PX / 8) + pp;
            V4<T> av[TM], bv[TN];
#pragma unroll
            for (int i = 0; i < TM; ++i) av[i] = lds4<T>(s_dz + (cgp + 4 * i) * WG_LD + p);
#pragma unroll
            for (int j = 0; j < TN; ++j) bv[j] = lds4<T>(s_y + (cg8 + 8 * j) * WG_LD + p);
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) dot4_acc(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
    // combine the 8 warps (each saw different pixels) in a fixed order, one partial tile per CTA
    T *red = s_dz;  // 8 * WG_TILE scalars <= (WG_CO + WG_CIT) * WG_LD
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) red[warp * WG_TILE + (cgp + 4 * i) * WG_CIT + cg8 + 8 * j] = acc[i][j];
    __syncthreads();
    for (int idx = threadIdx.x; idx < WG_TILE; idx += WG_THREADS) {
        T t = T(0);
#pragma unroll
        for (int w = 0; w < WG_THREADS / 32; ++w) t += red[w * WG_TILE + idx];
        a.partial[((int64_t)blockIdx.x * gridDim.y + tile) * WG_TILE + idx] = t;
    }
}

template <typename T>
struct GradLayer {
    const T *partial;
    const unsigned long long *accB;
    int PX, ntiles, tiles_cit, Cin, Cout, taps, wg_co, wg_cit;
    int64_t base;  // offset of this layer's first parameter (conv.weight, conv.bias, bn.weight, bn.bias follow each other)
};
template <typename T>
struct GradArgs {
    GradLayer<T> L[PNODE_CONV_MAX_LAYERS];
    int nl, accumulate, bn_grads;  // bn_grads = 0: the (global) BatchNorm gradients are contributed by rank 0 only
    int64_t np;
    const unsigned *flag;
    T *out;
    double coef;
};

// one group of G lanes per parameter: the lanes stride over the per-CTA partial tiles, then combine in a fixed order
template <typename T, int G>
__global__ void __launch_bounds__(256) grads_finalize_kernel(const GradArgs<T> a) {
    const int sub = threadIdx.x % G;
    const int64_t stride = (int64_t)gridDim.x * (blockDim.x / G);
    const int64_t rounds = (a.np + stride - 1) / stride;
    pdl::pdl_launch_dependents();
    pdl::pdl_wait();
    const double bad = __ldcg(a.flag) != 0u ? NAN : 0.0;
    for (int64_t rd = 0; rd < rounds; ++rd) {
        const int64_t i = rd * stride + (int64_t)blockIdx.x * (blockDim.x / G) + threadIdx.x / G;
        const bool live = i < a.np;
        double val = 0.0;
        if (live) {
            int k = 0;
            while (k + 1 < a.nl && i >= a.L[k + 1].base) ++k;
            const GradLayer<T> &l = a.L[k];
            int64_t loc = i - l.base;
            const int64_t nw = (int64_t)l.Cout * l.Cin * l.taps;
            if (loc < nw) {
                const int co = (int)(loc / (l.Cin * l.taps)), cit = (int)(loc % (l.Cin * l.taps));
                const int tile = (co / l.wg_co) * l.tiles_cit + cit / l.wg_cit;
                const int idx = (co % l.wg_co) * l.wg_cit + cit % l.wg_cit;
                const int64_t tsz = (int64_t)l.wg_co * l.wg_cit;
                for (int b = sub; b < l.PX; b += G) val += (double)__ldcg(l.partial + ((int64_t)b * l.ntiles + tile) * tsz + idx);
            } else if (loc < nw + l.Cout) {
                val = 0.0;  // conv bias under a BatchNorm: sum_p dz = 0 exactly
            } else if (sub == 0) {
                loc -= nw + l.Cout;  // bn.weight gradient = sum [y>0] g xhat, bn.bias gradient = sum [y>0] g
                val = loc < l.Cout ? acc128_read(l.accB, l.Cout, (int)loc, 1) : acc128_read(l.accB, l.Cout, (int)(loc - l.Cout), 0);
                val = a.bn_grads ? val + bad : 0.0;
            }
        }
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) val += __shfl_xor_sync(FULL, val, o);
        if (live && sub == 0) a.out[i] = a.accumulate ? (T)((double)a.out[i] + a.coef * val) : (T)val;
    }
}

#if PNODE_CB_PART != 2
// unit-test hook: every thread adds one value into ONE accumulator (all replicas used), then the total is read back
__global__ void acc128_probe_kernel(const double *__restrict__ v, int64_t n, unsigned long long *acc, unsigned *flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) acc128_add(acc + ((int64_t)(blockIdx.x % ACC_R) * 2) * 2, v[i], flag);
}
__global__ void acc128_read_kernel(const unsigned long long *acc, const unsigned *flag, double *out) {
    out[0] = *flag != 0u ? NAN : acc128_read(acc, 1, 0, 0);
}
#endif

// ---- host side ------------------------------------------------------------------------------------------------------------
struct CbPlan {
    int L, Cmax;
    int64_t M, Mglobal, npg;
    size_t esz;
    size_t off_z[PNODE_CONV_MAX_LAYERS], off_g[PNODE_CONV_MAX_LAYERS], off_accF[PNODE_CONV_MAX_LAYERS], off_accB[PNODE_CONV_MAX_LAYERS];
    size_t off_flag, off_acc0, acc_bytes, accB_bytes, off_wpart[PNODE_CONV_MAX_LAYERS], act_total, total;
    int kind[PNODE_CONV_MAX_LAYERS], taps[PNODE_CONV_MAX_LAYERS];
    int wg_px[PNODE_CONV_MAX_LAYERS], wg_tiles_cit[PNODE_CONV_MAX_LAYERS], wg_ntiles[PNODE_CONV_MAX_LAYERS];
    int wg_tm[PNODE_CONV_MAX_LAYERS], wg_tn[PNODE_CONV_MAX_LAYERS];
    int64_t pbase[PNODE_CONV_MAX_LAYERS + 1];
};

static size_t align_up(size_t v) { return (v + 255) & ~(size_t)255; }

struct ConvGrid {
    int rc, cg, gy, gx;
    size_t smem;
};

// One launcher for every kernel of this file: opt-in dynamic shared memory is raised once per kernel (not per launch), then
// pdl::launch_pdl launches it as a programmatic dependent launch.  Every kernel of this file lets its successor start early
// (its prologue -- barrier init, weight staging -- overlaps this kernel's tail) and waits for its predecessor's memory before
// touching anything that depends on it.
template <typename... KArgs, typename... Args>
static cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    static std::map<const void *, size_t> raised;
    if (smem > 48 * 1024 - 4096) {
        size_t &have = raised[reinterpret_cast<const void *>(kernel)];
        if (have < smem) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            have = smem;
        }
    }
    return pdl::launch_pdl(kernel, grid, block, smem, st, args...);
}

// thread = 4 pixels x rc output channels, CTA = 64 pixel groups x cg channel groups, grid.y = further channel tiles
static ConvGrid conv_grid(int CA, int CB, int taps, int ncoef_in, bool dgrad_epi, int64_t npg, size_t esz) {
    ConvGrid g;
    const int sm = sm_count();
    constexpr int occ = 1024;  // resident threads per SM the grid aims at
    g.rc = CB % 8 == 0 ? 8 : 4;
    int groups = CB / g.rc;
    g.cg = groups < CB_MAXCG ? groups : CB_MAXCG;
    while (groups % g.cg != 0) --g.cg;
    g.gy = groups / g.cg;
    const int tiles = (int)((npg + CB_PGX - 1) / CB_PGX);
    int cap = sm * (occ / (CB_PGX * g.cg)) / g.gy;
    if (cap < 1) cap = 1;
    g.gx = tiles < cap ? tiles : cap;
    g.smem = ((size_t)CA * taps * g.cg * g.rc + (size_t)ncoef_in * CA + (dgrad_epi ? 4 * g.cg * g.rc : 0)) * esz;
    return g;
}

static int cb_plan(const pnode_convblock_desc *d, CbPlan &p) {
    PNODE_REQUIRE(d != nullptr, "convblock: null descriptor");
    PNODE_REQUIRE(d->nlayers >= 1 && d->nlayers <= PNODE_CONV_MAX_LAYERS, "convblock: 1..%d layers (got %d)",
                  PNODE_CONV_MAX_LAYERS, d->nlayers);
    PNODE_REQUIRE(d->dtype == PNODE_F32 || d->dtype == PNODE_F64, "convblock: unsupported dtype %d", d->dtype);
    PNODE_REQUIRE(d->N >= 1 && d->H >= 1 && d->W >= 4 && d->W % 4 == 0 && (d->W & (d->W - 1)) == 0 && d->W <= 128,
                  "convblock: W must be a power of two in 4..128 (got N=%d H=%d W=%d)", d->N, d->H, d->W);
    p.L = d->nlayers;
    p.esz = d->dtype == PNODE_F32 ? 4 : 8;
    p.M = (int64_t)d->N * d->H * d->W;
    p.Mglobal = d->world > 1 && d->global_pixels > 0 ? d->global_pixels : p.M;
    p.npg = p.M / 4;
    p.Cmax = 0;
    p.pbase[0] = 0;
    for (int k = 0; k < p.L; ++k) {
        const pnode_conv_layer &l = d->layer[k];
        PNODE_REQUIRE(l.cin >= 4 && l.cout >= 4 && l.cin % 4 == 0 && l.cout % 4 == 0,
                      "convblock: channel counts must be multiples of 4 (layer %d: %d -> %d)", k, l.cin, l.cout);
        PNODE_REQUIRE(k == 0 || l.cin == d->layer[k - 1].cout, "convblock: layer %d input channels do not chain", k);
        if (l.kh == 1 && l.kw == 1 && l.ph == 0 && l.pw == 0) p.kind[k] = 0;
        else if (l.kh == 1 && l.kw == 3 && l.ph == 0 && l.pw == 1) p.kind[k] = 1;
        else if (l.kh == 3 && l.kw == 1 && l.ph == 1 && l.pw == 0) p.kind[k] = 2;
        else PNODE_REQUIRE(false, "convblock: layer %d kernel (%d,%d) pad (%d,%d) is not 1x1 / (1,3)p(0,1) / (3,1)p(1,0)", k,
                           l.kh, l.kw, l.ph, l.pw);
        PNODE_REQUIRE(l.d_weight && l.d_bias && l.d_gamma && l.d_beta, "convblock: layer %d has a null parameter", k);
        p.taps[k] = p.kind[k] == 0 ? 1 : 3;
        if (l.cin > p.Cmax) p.Cmax = l.cin;
        if (l.cout > p.Cmax) p.Cmax = l.cout;
        p.pbase[k + 1] = p.pbase[k] + (int64_t)l.cout * l.cin * p.taps[k] + 3 * (int64_t)l.cout;
    }
    PNODE_REQUIRE(p.Cmax <= 2048, "convblock: at most 2048 channels (got %d)", p.Cmax);
    PNODE_REQUIRE(d->world <= 1 || d->d_peer_bufs == nullptr || 4 * p.Cmax <= PNODE_PEER_NP_MAX,
                  "convblock: the in-kernel statistics exchange takes at most %d channels (got %d)", PNODE_PEER_NP_MAX / 4, p.Cmax);
    // activation region (one per saved evaluation): z_1..z_L, then the flag + forward accumulators (zeroed by one memset)
    size_t off = 0;
    for (int k = 0; k < p.L; ++k) {
        p.off_z[k] = off;
        off = align_up(off + (size_t)p.M * d->layer[k].cout * p.esz);
    }
    p.off_acc0 = off;
    p.off_flag = off;
    off += 256;
    for (int k = 0; k < p.L; ++k) {
        p.off_accF[k] = off;
        off += (size_t)ACC_R * d->layer[k].cout * 2 * 2 * sizeof(unsigned long long);
    }
    p.acc_bytes = off - p.off_acc0;
    p.act_total = align_up(off);
    // scratch region: backward accumulators (zeroed by one memset), g_k = dL/dy_k of every layer, weight-gradient partials
    off = 0;
    for (int k = 0; k < p.L; ++k) {
        p.off_accB[k] = off;
        off += (size_t)ACC_R * d->layer[k].cout * 2 * 2 * sizeof(unsigned long long);
    }
    p.accB_bytes = off;
    off = align_up(off);
    for (int k = 0; k < p.L; ++k) {
        p.off_g[k] = off;
        off = align_up(off + (size_t)p.M * d->layer[k].cout * p.esz);
    }
    const int sm = sm_count();
    for (int k = 0; k < p.L; ++k) {
        const pnode_conv_layer &l = d->layer[k];
        const ConvGrid f = conv_grid(l.cin, l.cout, p.taps[k], 2, false, p.npg, p.esz);
        const ConvGrid b = conv_grid(l.cout, l.cin, p.taps[k], 6, true, p.npg, p.esz);
        PNODE_REQUIRE(f.smem <= 200 * 1024 && b.smem <= 200 * 1024, "convblock: layer %d weights do not fit in shared memory", k);
        {  // gradient tile (4 TM) x (8 TN): least padding, then largest
            static const int cand[5][2] = {{4, 4}, {4, 6}, {8, 2}, {4, 3}, {2, 2}};
            const int rows = l.cout, cols = l.cin * p.taps[k];
            int64_t best = -1;
            for (int c = 0; c < 5; ++c) {
                const int co = 4 * cand[c][0], ci = 8 * cand[c][1];
                const int64_t area = (int64_t)((rows + co - 1) / co) * ((cols + ci - 1) / ci) * co * ci;
                if (best < 0 || area < best) best = area, p.wg_tm[k] = cand[c][0], p.wg_tn[k] = cand[c][1];
            }
        }
        const int wg_co = 4 * p.wg_tm[k], wg_cit = 8 * p.wg_tn[k];
        p.wg_tiles_cit[k] = (l.cin * p.taps[k] + wg_cit - 1) / wg_cit;
        p.wg_ntiles[k] = ((l.cout + wg_co - 1) / wg_co) * p.wg_tiles_cit[k];
        const int nchunks = (int)((p.npg + 31) / 32);
        constexpr int wg_occ = 2;  // CTAs per SM: measured best with the side stream (271 vs 289 us at 4)
        int px = sm * wg_occ / p.wg_ntiles[k];
        if (px < 1) px = 1;
        if (px > nchunks) px = nchunks;
        p.wg_px[k] = px;
    }
    for (int k = 0; k < p.L; ++k) {
        p.off_wpart[k] = off;
        off = align_up(off + (size_t)p.wg_px[k] * p.wg_ntiles[k] * (16 * p.wg_tm[k] * 2 * p.wg_tn[k]) * p.esz);
    }
    p.total = off;
    return 0;
}

struct PipeGrid {
    bool ok;
    int rc, cg, gy, gx, S, tiles;
    size_t smem;
};

// geometry of the pipelined kernel, or ok = false when the shape needs the direct kernel (halo rows, odd channel counts)
static PipeGrid pipe_grid(int kind, int src, int CA, int CB, int taps, int64_t npg, int HW, size_t esz) {
    PipeGrid g = {};
    constexpr int max_stages = 4, ctas_per_sm = 2;
    constexpr size_t smem_cap = 110 * 1024;  // per CTA, so that ctas_per_sm fit on an SM: stages are dropped (down to 2) first
    const int rcmax = esz == 8 ? 8 : 16;
    g.rc = 0;
    for (int rc = rcmax; rc >= (esz == 8 ? 4 : 8); rc >>= 1)
        if (CB % rc == 0) {
            g.rc = rc;
            break;
        }
    if (g.rc == 0) return g;
    const int groups = CB / g.rc;
    g.cg = groups % 2 == 0 ? 2 : 1;
    g.gy = groups / g.cg;
    const int PGT = CP_CONSUMERS / g.cg, TP = 4 * PGT;
    if (!((TP % HW == 0) || (HW % TP == 0 && kind != 2))) return g;
    const int KC = src == SRC_DZ ? 2 : 4, NT = src == SRC_DZ ? 2 : 1;
    if (CA % KC != 0) return g;
    const int ncoef = src == SRC_RAW ? 0 : (src == SRC_ACT ? 2 : 6);
    const int CT = g.cg * g.rc;
    const size_t head = (128 + ((size_t)CA * taps * CT + (size_t)ncoef * CA + 4 * CT) * esz + 127) & ~(size_t)127;
    const size_t stage = (size_t)NT * KC * TP * esz;
    g.S = max_stages;
    while (g.S > 2 && head + g.S * stage > smem_cap) --g.S;
    g.smem = head + g.S * stage;
    if (g.smem > 200 * 1024) return g;
    g.tiles = (int)((npg + PGT - 1) / PGT);
    int cap = sm_count() * ctas_per_sm / g.gy;
    if (cap < 1) cap = 1;
    g.gx = g.tiles < cap ? g.tiles : cap;
    g.ok = true;
    return g;
}

template <typename T, int KIND, int SRC, int EPI>
static int launch_conv_rc(const ConvArgs<T> &a_in, const ConvGrid &g, cudaStream_t st) {
    const PipeGrid pg = pipe_grid(KIND, SRC, a_in.CA, a_in.CB, KIND == 0 ? 1 : 3, a_in.npg, a_in.HW, sizeof(T));
    if (pg.ok) {
        ConvArgs<T> a = a_in;
        a.tiles = pg.tiles;
        dim3 grid(pg.gx, pg.gy);
#define PNODE_PIPE_LAUNCH(RC) \
    PNODE_CUDA_OK(launch_k(convp_kernel<T, KIND, SRC, EPI, RC>, grid, dim3(CP_CONSUMERS + 32), pg.smem, st, a, pg.cg, pg.S))
        if (pg.rc == 16) {
            if constexpr (sizeof(T) == 4) PNODE_PIPE_LAUNCH(16);
        } else if (pg.rc == 8) {
            PNODE_PIPE_LAUNCH(8);
        } else {
            if constexpr (sizeof(T) == 8) PNODE_PIPE_LAUNCH(4);
        }
#undef PNODE_PIPE_LAUNCH
        return 0;
    }
    const ConvArgs<T> &a = a_in;
    dim3 grid(g.gx, g.gy), block(CB_PGX, g.cg);
    if (g.rc == 8) PNODE_CUDA_OK(launch_k(conv_kernel<T, KIND, SRC, EPI, 8>, grid, block, g.smem, st, a));
    else PNODE_CUDA_OK(launch_k(conv_kernel<T, KIND, SRC, EPI, 4>, grid, block, g.smem, st, a));
    return 0;
}

template <typename T, int SRC, int EPI>
static int launch_conv(int kind, const ConvArgs<T> &a, const ConvGrid &g, cudaStream_t st) {
    if (kind == 0) return launch_conv_rc<T, 0, SRC, EPI>(a, g, st);
    if (kind == 1) return launch_conv_rc<T, 1, SRC, EPI>(a, g, st);
    return launch_conv_rc<T, 2, SRC, EPI>(a, g, st);
}

template <typename T, int KIND, int YSRC, int TM, int TN>
static int launch_wgrad_tile(const WgradArgs<T> &a, int px, int ntiles, cudaStream_t st) {
    const size_t smem = ((size_t)(4 * TM + 8 * TN) * WG_LD + 6 * 4 * TM + 2 * 8 * TN) * sizeof(T);
    PNODE_CUDA_OK(launch_k(conv_wgrad_kernel<T, KIND, YSRC, TM, TN>, dim3(px, ntiles), dim3(WG_THREADS), smem, st, a));
    return 0;
}

template <typename T, int KIND, int YSRC>
static int launch_wgrad_kind(int tm, int tn, const WgradArgs<T> &a, int px, int ntiles, cudaStream_t st) {
    if (tm == 4 && tn == 4) return launch_wgrad_tile<T, KIND, YSRC, 4, 4>(a, px, ntiles, st);
    if (tm == 4 && tn == 6) return launch_wgrad_tile<T, KIND, YSRC, 4, 6>(a, px, ntiles, st);
    if (tm == 8 && tn == 2) return launch_wgrad_tile<T, KIND, YSRC, 8, 2>(a, px, ntiles, st);
    if (tm == 4 && tn == 3) return launch_wgrad_tile<T, KIND, YSRC, 4, 3>(a, px, ntiles, st);
    return launch_wgrad_tile<T, KIND, YSRC, 2, 2>(a, px, ntiles, st);
}

template <typename T, int YSRC>
static int launch_wgrad(int kind, int tm, int tn, const WgradArgs<T> &a, int px, int ntiles, cudaStream_t st) {
    if (kind == 0) return launch_wgrad_kind<T, 0, YSRC>(tm, tn, a, px, ntiles, st);
    if (kind == 1) return launch_wgrad_kind<T, 1, YSRC>(tm, tn, a, px, ntiles, st);
    return launch_wgrad_kind<T, 2, YSRC>(tm, tn, a, px, ntiles, st);
}

// The weight-gradient kernel of a layer and its data-gradient kernel read the same inputs and do not depend on each other:
// the weight gradients run on a side stream (fork after the kernel that completed the layer's backward sums, join before the
// final gradient kernel), so the two latency-bound kernels share the SMs instead of queueing.
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork[PNODE_CONV_MAX_LAYERS + 1] = {}, join = nullptr;
    bool ok = false;
};
static SideStream &side_stream() {
    static SideStream s;
    static bool tried = false;
    if (!tried) {
        tried = true;
        bool ok = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) == cudaSuccess;
        for (int i = 0; ok && i <= PNODE_CONV_MAX_LAYERS; ++i) ok = cudaEventCreateWithFlags(&s.fork[i], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) == cudaSuccess;
        s.ok = ok;
    }
    return s;
}

template <typename T>
struct Bufs {
    unsigned char *a, *w;  // activation region, scratch region
    const CbPlan &p;
    Bufs(void *act, void *work, const CbPlan &pl) : a(static_cast<unsigned char *>(act)), w(static_cast<unsigned char *>(work)), p(pl) {}
    T *z(int k) const { return reinterpret_cast<T *>(a + p.off_z[k]); }
    unsigned long long *accF(int k) const { return reinterpret_cast<unsigned long long *>(a + p.off_accF[k]); }
    unsigned *flag() const { return reinterpret_cast<unsigned *>(a + p.off_flag); }
    T *g(int k) const { return reinterpret_cast<T *>(w + p.off_g[k]); }
    unsigned long long *accB(int k) const { return w ? reinterpret_cast<unsigned long long *>(w + p.off_accB[k]) : nullptr; }
    T *wpart(int k) const { return reinterpret_cast<T *>(w + p.off_wpart[k]); }
};

template <typename T>
static BnRef bn_ref(const pnode_convblock_desc *d, const Bufs<T> &b, int k) {
    const pnode_conv_layer &l = d->layer[k];
    BnRef r;
    r.accF = b.accF(k), r.accB = b.accB(k);
    r.gamma = l.d_gamma, r.beta = l.d_beta;
    r.rmean = l.d_running_mean, r.rvar = l.d_running_var;
    r.nbt = static_cast<long long *>(l.d_num_batches_tracked);
    r.eps = l.eps, r.momentum = l.momentum;
    r.C = l.cout;
    return r;
}

template <typename T>
static void fill_common(ConvArgs<T> &a, const pnode_convblock_desc *d, const CbPlan &p, const Bufs<T> &b) {
    a.H = d->H, a.W = d->W, a.HW = d->H * d->W;
    a.npg = p.npg;
    a.tiles = (int)((p.npg + CB_PGX - 1) / CB_PGX);
    a.M = (double)p.Mglobal;
    a.flag = b.flag();
    a.ticket = b.flag() + 16;
    a.peer_bufs = d->world > 1 ? reinterpret_cast<const unsigned long long *>(d->d_peer_bufs) : nullptr;
    a.rank = d->rank, a.world = d->world;
}

// z_1 .. z_L of the chain, the exact batch statistics of every layer, and the running-statistics updates of layers 1..L-1
// (layer L's update belongs to whoever consumes z_L next: act_out_kernel or top_stats_kernel)
template <typename T>
static int forward_chain(const pnode_convblock_desc *d, const CbPlan &p, const Bufs<T> &b, const T *x, unsigned long long &epoch,
                         cudaStream_t st) {
    PNODE_CUDA_OK(cudaMemsetAsync(b.a + p.off_acc0, 0, p.acc_bytes, st));
    for (int k = 0; k < p.L; ++k) {
        const pnode_conv_layer &l = d->layer[k];
        ConvArgs<T> a = {};
        fill_common(a, d, p, b);
        a.in = k == 0 ? x : b.z(k - 1);
        if (k > 0) a.bin = bn_ref(d, b, k - 1), a.upd_in = 1;
        a.w = static_cast<const T *>(l.d_weight), a.bias = static_cast<const T *>(l.d_bias);
        a.out = b.z(k);
        a.acc_out = b.accF(k);
        a.epoch = epoch++;
        a.CA = l.cin, a.CB = l.cout;
        const ConvGrid g = conv_grid(l.cin, l.cout, p.taps[k], k == 0 ? 0 : 2, false, p.npg, p.esz);
        int rc = k == 0 ? launch_conv<T, SRC_RAW, EPI_FWD>(p.kind[k], a, g, st) : launch_conv<T, SRC_ACT, EPI_FWD>(p.kind[k], a, g, st);
        if (rc) return rc;
    }
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

template <typename T>
static int act_out(const pnode_convblock_desc *d, const CbPlan &p, const Bufs<T> &b, T *out, const T *base, double base_coef,
                   double kcoef, T *kout, cudaStream_t st) {
    const int C = d->layer[p.L - 1].cout;
    const int64_t nvec = p.M * C / 4;
    int64_t blocks = (nvec + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    PNODE_CUDA_OK(launch_k(act_out_kernel<T>, dim3((unsigned)blocks), dim3(256), 2 * C * sizeof(T), st, (const T *)b.z(p.L - 1),
                           bn_ref(d, b, p.L - 1), (double)p.Mglobal, (const unsigned *)b.flag(), 1, d->H * d->W, nvec, out, base,
                           (T)base_coef, (T)kcoef, kout));
    return 0;
}

template <typename T>
static int vjp_chain(const pnode_convblock_desc *d, const CbPlan &p, const Bufs<T> &b, const T *x, const T *w, T *vu, T *gout,
                     double coef, int accumulate, int replay_running, unsigned long long &epoch, cudaStream_t st) {
    const int L = p.L;
    PNODE_CUDA_OK(cudaMemsetAsync(b.w + p.off_accB[0], 0, p.accB_bytes, st));
    {  // BatchNorm-backward sums of the top layer
        const pnode_conv_layer &l = d->layer[L - 1];
        ConvArgs<T> a = {};
        fill_common(a, d, p, b);
        a.in = w, a.zprev = b.z(L - 1);
        a.bout = bn_ref(d, b, L - 1), a.upd_out = 1;
        a.acc_out = b.accB(L - 1);
        a.epoch = epoch++;
        a.CA = 0, a.CB = l.cout;
        const ConvGrid g = conv_grid(0, l.cout, 1, 0, true, p.npg, p.esz);
        dim3 grid(g.gx, g.gy), block(CB_PGX, g.cg);
        const size_t smem = (size_t)4 * g.cg * g.rc * sizeof(T);
        if (g.rc == 8) PNODE_CUDA_OK(launch_k(top_stats_kernel<T, 8>, grid, block, smem, st, a));
        else PNODE_CUDA_OK(launch_k(top_stats_kernel<T, 4>, grid, block, smem, st, a));
    }
    const T *gk = w;
    SideStream &side = side_stream();
    const bool fork = side.ok && gout != nullptr;
    for (int k = L - 1; k >= 0; --k) {
        const pnode_conv_layer &l = d->layer[k];
        cudaStream_t wst = st;
        if (fork) {  // everything wgrad_k needs (g_k, the backward sums of layer k) is complete at this point of the main stream
            PNODE_CUDA_OK(cudaEventRecord(side.fork[k], st));
            PNODE_CUDA_OK(cudaStreamWaitEvent(side.stream, side.fork[k], 0));
            wst = side.stream;
        }
        if (gout != nullptr) {
            WgradArgs<T> wa = {};
            wa.g = gk, wa.z = b.z(k), wa.bk = bn_ref(d, b, k);
            wa.yin = k == 0 ? x : b.z(k - 1);
            if (k > 0) wa.bin = bn_ref(d, b, k - 1);
            wa.flag = b.flag();
            wa.partial = b.wpart(k);
            wa.Cin = l.cin, wa.Cout = l.cout, wa.H = d->H, wa.W = d->W, wa.HW = d->H * d->W;
            wa.tiles_cit = p.wg_tiles_cit[k];
            wa.npg = p.npg;
            wa.nchunks = (int)((p.npg + 31) / 32);
            wa.M = (double)p.Mglobal;
            int rc = k == 0 ? launch_wgrad<T, SRC_RAW>(p.kind[k], p.wg_tm[k], p.wg_tn[k], wa, p.wg_px[k], p.wg_ntiles[k], wst)
                            : launch_wgrad<T, SRC_ACT>(p.kind[k], p.wg_tm[k], p.wg_tn[k], wa, p.wg_px[k], p.wg_ntiles[k], wst);
            if (rc) return rc;
        }
        if (k == 0 && vu == nullptr) break;
        ConvArgs<T> a = {};
        fill_common(a, d, p, b);
        a.in = gk, a.in2 = b.z(k), a.bin = bn_ref(d, b, k);
        a.w = static_cast<const T *>(l.d_weight);
        a.CA = l.cout, a.CB = l.cin;
        const ConvGrid g = conv_grid(l.cout, l.cin, p.taps[k], 6, k > 0, p.npg, p.esz);
        int rc;
        if (k == 0) {
            a.out = vu;
            rc = launch_conv<T, SRC_DZ, EPI_NONE>(p.kind[k], a, g, st);
        } else {
            a.out = b.g(k - 1);
            a.zprev = b.z(k - 1), a.bout = bn_ref(d, b, k - 1);
            a.upd_out = replay_running;  // saved activations: the module's forward re-evaluation still advances the buffers
            a.acc_out = b.accB(k - 1);
            a.epoch = epoch++;
            rc = launch_conv<T, SRC_DZ, EPI_DGRAD>(p.kind[k], a, g, st);
            gk = a.out;
        }
        if (rc) return rc;
    }
    if (fork) {
        PNODE_CUDA_OK(cudaEventRecord(side.join, side.stream));
        PNODE_CUDA_OK(cudaStreamWaitEvent(st, side.join, 0));
    }
    if (gout != nullptr) {
        GradArgs<T> ga = {};
        ga.nl = L, ga.accumulate = accumulate, ga.np = p.pbase[L], ga.out = gout, ga.coef = coef, ga.flag = b.flag();
        ga.bn_grads = d->world <= 1 || d->d_peer_bufs == nullptr || d->rank == 0;
        int pxmax = 1;
        for (int k = 0; k < L; ++k) {
            ga.L[k].partial = b.wpart(k), ga.L[k].accB = b.accB(k);
            ga.L[k].PX = p.wg_px[k], ga.L[k].ntiles = p.wg_ntiles[k], ga.L[k].tiles_cit = p.wg_tiles_cit[k];
            ga.L[k].Cin = d->layer[k].cin, ga.L[k].Cout = d->layer[k].cout, ga.L[k].taps = p.taps[k];
            ga.L[k].base = p.pbase[k];
            ga.L[k].wg_co = 4 * p.wg_tm[k], ga.L[k].wg_cit = 8 * p.wg_tn[k];
            pxmax = p.wg_px[k] > pxmax ? p.wg_px[k] : pxmax;
        }
        const int G = pxmax > 8 ? 32 : 4;
        int64_t blocks = (ga.np * G + 255) / 256;
        const int64_t cap = (int64_t)sm_count() * 8;
        if (blocks > cap) blocks = cap;
        if (G == 32) PNODE_CUDA_OK(launch_k(grads_finalize_kernel<T, 32>, dim3((unsigned)blocks), dim3(256), 0, st, ga));
        else PNODE_CUDA_OK(launch_k(grads_finalize_kernel<T, 4>, dim3((unsigned)blocks), dim3(256), 0, st, ga));
    }
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

static bool cb_aligned(const void *p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// one non-template entry per scalar type, so that the two types can live in two objects
template <typename T>
static int run_forward(const pnode_convblock_desc *desc, const CbPlan &p, const void *d_x, void *d_out, const void *d_base,
                       double base_coef, double k_coef, void *d_k, void *d_act, cudaStream_t st) {
    unsigned long long epoch = desc->epoch;
    Bufs<T> b(d_act, nullptr, p);
    int rc = forward_chain<T>(desc, p, b, static_cast<const T *>(d_x), epoch, st);
    if (rc) return rc;
    return act_out<T>(desc, p, b, static_cast<T *>(d_out), static_cast<const T *>(d_base), base_coef, k_coef, static_cast<T *>(d_k), st);
}

template <typename T>
static int run_vjp(const pnode_convblock_desc *desc, const CbPlan &p, const void *d_x, const void *d_w, void *d_vu, void *d_grads,
                   double coef, int accumulate, void *d_act, int act_valid, void *d_work, cudaStream_t st) {
    unsigned long long epoch = desc->epoch;
    Bufs<T> b(d_act, d_work, p);
    if (!act_valid) {
        int rc = forward_chain<T>(desc, p, b, static_cast<const T *>(d_x), epoch, st);
        if (rc) return rc;
    }
    return vjp_chain<T>(desc, p, b, static_cast<const T *>(d_x), static_cast<const T *>(d_w), static_cast<T *>(d_vu),
                        static_cast<T *>(d_grads), coef, accumulate, act_valid != 0, epoch, st);
}

int convblock_forward_f64(const pnode_convblock_desc *desc, const void *d_x, void *d_out, const void *d_base, double base_coef,
                          double k_coef, void *d_k, void *d_act, void *stream);
int convblock_vjp_f64(const pnode_convblock_desc *desc, const void *d_x, const void *d_w, void *d_vu, void *d_grads, double coef,
                      int accumulate, void *d_act, int act_valid, void *d_work, void *stream);

#if PNODE_CB_PART != 1
int convblock_forward_f64(const pnode_convblock_desc *desc, const void *d_x, void *d_out, const void *d_base, double base_coef,
                          double k_coef, void *d_k, void *d_act, void *stream) {
    CbPlan p;
    int rc = cb_plan(desc, p);
    if (rc) return rc;
    return run_forward<double>(desc, p, d_x, d_out, d_base, base_coef, k_coef, d_k, d_act, static_cast<cudaStream_t>(stream));
}
int convblock_vjp_f64(const pnode_convblock_desc *desc, const void *d_x, const void *d_w, void *d_vu, void *d_grads, double coef,
                      int accumulate, void *d_act, int act_valid, void *d_work, void *stream) {
    CbPlan p;
    int rc = cb_plan(desc, p);
    if (rc) return rc;
    return run_vjp<double>(desc, p, d_x, d_w, d_vu, d_grads, coef, accumulate, d_act, act_valid, d_work,
                           static_cast<cudaStream_t>(stream));
}
#endif

}  // namespace pnode

#if PNODE_CB_PART != 2
using namespace pnode;

extern "C" {

int pnode_acc128_probe(const double *d_values, int64_t n, double *d_out, void *d_work, void *stream) {
    PNODE_REQUIRE(d_values && d_out && d_work && n >= 0, "pnode_acc128_probe: null argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned long long *acc = static_cast<unsigned long long *>(d_work);
    unsigned *flag = reinterpret_cast<unsigned *>(acc + ACC_R * 2 * 2);
    PNODE_CUDA_OK(cudaMemsetAsync(d_work, 0, 256, st));
    if (n > 0) acc128_probe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_values, n, acc, flag);
    acc128_read_kernel<<<1, 1, 0, st>>>(acc, flag, d_out);
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

int64_t pnode_convblock_act_bytes(const pnode_convblock_desc *desc) {
    CbPlan p;
    if (cb_plan(desc, p) != 0) return -1;
    return (int64_t)p.act_total;
}

int64_t pnode_convblock_work_bytes(const pnode_convblock_desc *desc) {
    CbPlan p;
    if (cb_plan(desc, p) != 0) return -1;
    return (int64_t)p.total;
}

int64_t pnode_convblock_param_count(const pnode_convblock_desc *desc) {
    CbPlan p;
    if (cb_plan(desc, p) != 0) return -1;
    return p.pbase[p.L];
}

int pnode_convblock_forward(const pnode_convblock_desc *desc, const void *d_x, void *d_out, const void *d_base,
                            double base_coef, double k_coef, void *d_k, void *d_act, void *stream) {
    CbPlan p;
    int rc = cb_plan(desc, p);
    if (rc) return rc;
    PNODE_REQUIRE(d_x && d_act && (d_out || d_k), "pnode_convblock_forward: null argument");
    PNODE_REQUIRE(cb_aligned(d_x) && cb_aligned(d_out) && cb_aligned(d_base) && cb_aligned(d_k) && cb_aligned(d_act),
                  "pnode_convblock_forward: tensors must be 16-byte aligned");
    PNODE_REQUIRE(desc->layer[p.L - 1].cout == desc->layer[0].cin, "pnode_convblock_forward: an ODE right-hand side maps C -> C");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (desc->dtype == PNODE_F32) return run_forward<float>(desc, p, d_x, d_out, d_base, base_coef, k_coef, d_k, d_act, st);
    return convblock_forward_f64(desc, d_x, d_out, d_base, base_coef, k_coef, d_k, d_act, st);
}

int pnode_convblock_vjp(const pnode_convblock_desc *desc, const void *d_x, const void *d_w, void *d_vu, void *d_grads,
                        double coef, int accumulate, void *d_act, int act_valid, void *d_work, void *stream) {
    CbPlan p;
    int rc = cb_plan(desc, p);
    if (rc) return rc;
    PNODE_REQUIRE(d_x && d_w && d_act && d_work && (d_vu || d_grads), "pnode_convblock_vjp: null argument");
    PNODE_REQUIRE(cb_aligned(d_x) && cb_aligned(d_w) && cb_aligned(d_vu) && cb_aligned(d_act) && cb_aligned(d_work),
                  "pnode_convblock_vjp: tensors must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (desc->dtype == PNODE_F32)
        return run_vjp<float>(desc, p, d_x, d_w, d_vu, d_grads, coef, accumulate, d_act, act_valid, d_work, st);
    return convblock_vjp_f64(desc, d_x, d_w, d_vu, d_grads, coef, accumulate, d_act, act_valid, d_work, st);
}

}  // extern "C"
#endif
