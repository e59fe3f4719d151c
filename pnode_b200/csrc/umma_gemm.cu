// Tensor-core matrix products for the wide right-hand sides (SINODE MLP, implicit-stage inverse apply, GEMM-sized conv
// layers): TMA-fed tcgen05.mma with the accumulators in tensor memory, hand-written for sm_100a.
//
// The state is fp64 (reference: PETSc scalar type, tests/test_pnode.py:127-130) or fp32, and results must match the
// reference to 1e-10 / 1e-4.  The 5th-generation tensor cores have no fp64 mode and TF32 alone is 1e-3, so every
// operand is a SLICED matrix and a product is a short sum of exact slice products:
//
//   kind i8   (fp64):  x[r][k] = 2^e[r] * sum_s q_s[r][k] 2^-(6+8s),  q_s signed bytes (balanced base-256 digits),
//              S = 6 slices (46 bits).
//              A.B^T = 2^(ea+eb) * sum_{d<S} 2^-(12+8d) * sum_{i+j=d} (q^A_i . q^B_j)      [Ozaki splitting]
//              every slice product is an EXACT int32 dot product (tcgen05.mma kind::i8), one TMEM accumulator per
//              diagonal d; the fp64 combination happens once, in the epilogue.  A diagonal sums up to 6 pairs of
//              digits per reduction index, so the int32 accumulators (which wrap: no saturation) bound K <= 16384.
//   kind i8x  (fp64):  8 signed base-128 digits in [-64, 64] (55 bits); diagonal 7 reaches 8 * 64 * 64 * K, which
//              fits int32 up to K = 65535.
//   kind tf32 (fp32):  x = hi + lo, hi = tf32(x), lo = x - hi;  A.B^T = hi.hi + hi.lo + lo.hi  (3xTF32, fp32 accumulate
//              in TMEM), relative error ~2^-21 per product.
//
// One CTA computes a 128 x BN tile of C: warp 4 (one lane) issues the TMA loads of ALL slices of the current K block
// into a ring of shared-memory stages (3-d tensor maps {K, rows, slice}, hardware swizzle, zero fill outside the
// matrix), warp 5 (one lane) issues the tcgen05.mma of every slice pair i+j<S against those tiles -- each slice tile is
// read from shared memory S times but fetched from L2 once -- and warps 0-3 drain the accumulators with tcgen05.ld,
// combine / scale / add bias / ReLU / mask / accumulate and store.
#include <cuda.h>

#include "common.cuh"
#include "umma.cuh"

namespace pnode {
namespace umma {

template <int KIND>
struct Cfg;
template <>
struct Cfg<KIND_I8> {  // dense digits: base 256, balanced (all signed bytes) -> 21 slice pairs for 46 bits
    static constexpr int S = PNODE_I8_SLICES, BN = 64, KB = 64, STAGES = 3, NACC = PNODE_I8_SLICES, ELEM = 1;
    static constexpr bool INT = true, DENSE = true;
    static constexpr int BASE_BITS = 8, LEAD_BITS = 6;  // digit width; magnitude bits of the leading digit
    using Out = double;
};
template <>
struct Cfg<KIND_I8X> {  // one more slice (55 bits): products with heavy cancellation (stiff inverse apply)
    static constexpr int S = PNODE_I8X_SLICES, BN = 64, KB = 64, STAGES = 2, NACC = PNODE_I8X_SLICES, ELEM = 1;
    static constexpr bool INT = true, DENSE = false;  // signed digits in [-64, 64] (base 128): K <= PNODE_I8X_MAX_K
    static constexpr int BASE_BITS = 7, LEAD_BITS = 6;
    using Out = double;
};
template <>
struct Cfg<KIND_TF32> {
    static constexpr int S = 2, BN = 64, KB = 128, STAGES = 4, NACC = 1, ELEM = 4;
    static constexpr bool INT = false, DENSE = false;
    static constexpr int BASE_BITS = 0, LEAD_BITS = 0;
    using Out = float;
};


// ---- PTX wrappers ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol error traps after ~2 s instead of hanging the device.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000ll) asm volatile("trap;");
    }
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
template <int KIND>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    if constexpr (Cfg<KIND>::INT) {
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}" ::"r"(
                         tmem_d),
                     "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
                     : "memory");
    } else {
        asm volatile(
            "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
            : "memory");
    }
}
__device__ __forceinline__ void tc_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor of a K-major tile whose rows are KB bytes (= the swizzle span) and dense:
// 8-row groups are 8*KB bytes apart (SBO); LBO is unused for swizzled K-major operands; version 1 = sm_100.
template <int KB>
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr) {
    uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((8 * KB) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(KB == 128 ? 2 : (KB == 64 ? 4 : 6)) << 61;
    return d;
}

// Instruction descriptor (dense, K-major A and B, M = 128, N = BN).  Integer kinds: per-operand signedness.
template <int KIND, int BN>
__device__ __forceinline__ constexpr uint32_t instr_desc(bool a_signed = true, bool b_signed = true) {
    uint32_t fmt = Cfg<KIND>::INT ? ((2u << 4) | ((a_signed ? 1u : 0u) << 7) | ((b_signed ? 1u : 0u) << 10))  // D = S32
                                  : ((1u << 4) | (2u << 7) | (2u << 10));                                   // D = F32, TF32
    return fmt | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

__device__ __forceinline__ double pow2(int e) {  // 2^e, |e| < 1000
    return __longlong_as_double((long long)(1023 + e) << 52);
}

// ---- the kernel -----------------------------------------------------------------------------------------------------
constexpr int EPI_WARPS = 16;                    // 4 per TMEM lane quarter: the epilogue arithmetic is latency bound with one
constexpr int GEMM_THREADS = 32 * (EPI_WARPS + 2);  // warp per scheduler; + one TMA-producer warp + one MMA-issuer warp
constexpr int TMA_THREAD = 32 * EPI_WARPS, MMA_THREAD = 32 * (EPI_WARPS + 1);

template <int KIND>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
    umma_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, int M, int N,
                     int K, Epilogue ep) {
    using C = Cfg<KIND>;
    using Out = typename C::Out;
    constexpr int S = C::S, BN = C::BN, KB = C::KB, STAGES = C::STAGES;
    constexpr int A_TILE = 128 * KB, B_TILE = BN * KB, STAGE_BYTES = S * (A_TILE + B_TILE);
    constexpr int TMEM_COLS = (C::NACC * BN <= 32) ? 32 : (C::NACC * BN <= 64) ? 64 : (C::NACC * BN <= 128) ? 128
                              : (C::NACC * BN <= 256) ? 256 : 512;
    static_assert(C::NACC * BN <= 512, "accumulators exceed tensor memory");

    pdl_launch_dependents();
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + STAGES * STAGE_BYTES);
    uint64_t *empty = full + STAGES;
    uint64_t *accfull = empty + STAGES;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(accfull + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.y * 128, n0 = blockIdx.x * BN;
    // split-K: grid.z slices of kb_per_split K blocks each, every slice writes its own output (C + z * split_stride)
    const int total_kb = (K * C::ELEM + KB - 1) / KB;
    const int kb_begin = ep.kb_per_split > 0 ? (int)blockIdx.z * ep.kb_per_split : 0;
    const int num_kb = ep.kb_per_split > 0 ? max(0, min(ep.kb_per_split, total_kb - kb_begin)) : total_kb;

    if (threadIdx.x == TMA_THREAD) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(accfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"((uint32_t)TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_wait();  // barriers, tensor memory and descriptors are set up: from here on the predecessors' results are needed
    const uint32_t tmem_base = *tmem_slot;

    if (threadIdx.x == TMA_THREAD) {
        // ---- TMA producer: all slices of K block kb into stage kb % STAGES ----
        for (int kb = 0; kb < num_kb; ++kb) {
            const int st = kb % STAGES, it = kb / STAGES;
            if (kb >= STAGES) mbar_wait(&empty[st], (it - 1) & 1);
            uint8_t *sa = smem + st * STAGE_BYTES, *sb = sa + S * A_TILE;
            mbar_expect_tx(&full[st], STAGE_BYTES);
            const int k0 = (kb_begin + kb) * (KB / C::ELEM);
#pragma unroll
            for (int s = 0; s < S; ++s) tma_load_3d(sa + s * A_TILE, &map_a, &full[st], k0, m0, s);
#pragma unroll
            for (int s = 0; s < S; ++s) tma_load_3d(sb + s * B_TILE, &map_b, &full[st], k0, n0, s);
        }
    } else if (threadIdx.x == MMA_THREAD) {
        // ---- MMA issuer: every slice pair i + j < S of this K block ----
        for (int kb = 0; kb < num_kb; ++kb) {
            const int st = kb % STAGES, it = kb / STAGES;
            mbar_wait(&full[st], it & 1);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + st * STAGE_BYTES), sb = sa + S * A_TILE;
#pragma unroll
            for (int k = 0; k < KB / 32; ++k) {
#pragma unroll
                for (int d = 0; d < S; ++d) {
#pragma unroll
                    for (int i = 0; i <= d; ++i) {
                        const int j = d - i;
                        const uint64_t ad = smem_desc<KB>(sa + i * A_TILE) + (uint64_t)(k * 2);
                        const uint64_t bd = smem_desc<KB>(sb + j * B_TILE) + (uint64_t)(k * 2);
                        const int acc = C::INT ? d : 0;
                        const bool first = (kb == 0) && (k == 0) && (i == 0) && (C::INT || d == 0);
                        constexpr uint32_t idesc = instr_desc<KIND, BN>();
                        tc_mma<KIND>(tmem_base + acc * BN, ad, bd, idesc, first ? 0u : 1u);
                    }
                }
            }
            tc_commit(&empty[st]);  // frees the stage when these MMAs have read it
        }
        tc_commit(accfull);
    } else if (warp < EPI_WARPS) {
        // ---- epilogue: warp = TMEM lane quarter (warp % 4: a warp may only touch its own 32 lanes) x column group
        // (warp / 4).  Phase 1: thread = one row: combine the diagonals, scale by the row exponent, park the values in shared
        // memory (the pipeline stages are free once the last MMA has completed).  Phase 2: lanes along the columns, CW
        // columns of 32 / CW rows per step: coalesced bias / mask / accumulate / store, loads batched for latency.
        if (num_kb > 0) {
            mbar_wait(accfull, 0);
            tc_fence_after();
        }
        constexpr int G = EPI_WARPS / 4, CW = BN / G;  // column groups, columns per group
        static_assert(CW % 8 == 0 && CW <= 32 && 32 % CW == 0, "epilogue column split");
        constexpr int TP = BN + 1;  // row pitch of the parked tile (elements): conflict-free for both phases
        static_assert(128 * TP * (int)sizeof(Out) <= STAGE_BYTES, "parked tile does not fit one pipeline stage");
        const int quarter = warp & 3, cg = warp >> 2;
        Out *tile = reinterpret_cast<Out *>(smem) + (quarter * 32) * TP + cg * CW;
        const int mrow0 = m0 + quarter * 32;
        const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16);
        double srow = 1.0;
        if constexpr (C::INT) srow = (mrow0 + lane < M) ? pow2(ep.ea[mrow0 + lane]) : 0.0;
#pragma unroll
        for (int c0 = 0; c0 < CW; c0 += 8) {
            double v[8];
            if constexpr (C::INT) {
                uint32_t r[S][8];
#pragma unroll
                for (int d = 0; d < S; ++d) tc_ld8(trow + d * BN + cg * CW + c0, r[d]);
                tc_wait_ld();
                if (num_kb == 0) {
#pragma unroll
                    for (int d = 0; d < S; ++d)
#pragma unroll
                        for (int q = 0; q < 8; ++q) r[d][q] = 0u;
                }
                // diagonal d carries weight 2^-(2 LEAD + BASE d): Horner in int64, in two halves that each stay below 2^53
                constexpr int NH = C::DENSE ? (S < 3 ? S : 3) : (S < 4 ? S : 4);
                constexpr long long RADIX = 1ll << C::BASE_BITS;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    long long hi = 0, lo = 0;
#pragma unroll
                    for (int d = 0; d < NH; ++d) hi = hi * RADIX + (long long)(int)r[d][q];
#pragma unroll
                    for (int d = NH; d < S; ++d) lo = lo * RADIX + (long long)(int)r[d][q];
                    double x = (double)hi * pow2(-(2 * C::LEAD_BITS + C::BASE_BITS * (NH - 1)));
                    if (S > NH) x = fma((double)lo, pow2(-(2 * C::LEAD_BITS + C::BASE_BITS * (S - 1))), x);
                    v[q] = x * srow;
                }
            } else {
                uint32_t r[8];
                tc_ld8(trow + cg * CW + c0, r);
                tc_wait_ld();
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] = num_kb == 0 ? 0.0 : (double)__uint_as_float(r[q]);
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) tile[lane * TP + c0 + q] = (Out)v[q];
        }
        __syncwarp();
        constexpr int RPS = 32 / CW;                 // rows per step
        const int col = lane % CW, rsub = lane / CW; // this lane's column within the group / row within the step
        const int n = n0 + cg * CW + col;
        const bool ncol = n < N;
        double scol = 1.0, bcol = 0.0;
        if (ncol) {
            if constexpr (C::INT) scol = pow2(ep.eb[n]);
            if (ep.bias) bcol = (double)reinterpret_cast<const Out *>(ep.bias)[n];
        }
        double ma = 1.0, mb = 0.0, qa = 0.0, qb = 0.0;  // mask kept where ma * mask + mb > 0;  q = qa * mask + qb
        if (ncol) {
            if (ep.mask_a) ma = (double)reinterpret_cast<const Out *>(ep.mask_a)[n];
            if (ep.mask_b) mb = (double)reinterpret_cast<const Out *>(ep.mask_b)[n];
            if (ep.stat_mode == 2) {
                qa = (double)reinterpret_cast<const Out *>(ep.q_a)[n];
                qb = (double)reinterpret_cast<const Out *>(ep.q_b)[n];
            }
        }
        double st1 = 0.0, st2 = 0.0;  // column statistics of the stored values (this lane's rows)
        Out *cbase = reinterpret_cast<Out *>(ep.C) + (ep.kb_per_split > 0 ? (long long)blockIdx.z * ep.split_stride : 0);
        const int rows = min(32, M - mrow0);
        constexpr int UN = 8;
        for (int rb = 0; rb < rows; rb += RPS * UN) {
            double acc[UN], msk[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) {           // all global loads of the batch first
                const int r = rb + u * RPS + rsub;
                acc[u] = 0.0, msk[u] = 1.0;
                if (ncol && r < rows) {
                    const long long m = mrow0 + r;
                    if (ep.accumulate) acc[u] = (double)cbase[m * ep.ldc + n];
                    if (ep.mask) msk[u] = (double)reinterpret_cast<const Out *>(ep.mask)[m * ep.ldmask + n];
                }
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int r = rb + u * RPS + rsub;
                if (ncol && r < rows) {
                    double x = ((double)tile[r * TP + col] * scol + bcol) * ep.alpha;
                    if (ep.relu) x = x > 0.0 ? x : 0.0;
                    x = (ma * msk[u] + mb) > 0.0 ? x : 0.0;
                    const Out stored = (Out)(x + acc[u]);
                    cbase[(long long)(mrow0 + r) * ep.ldc + n] = stored;
                    if (ep.stat_mode) {
                        const double sv = (double)stored;
                        st1 += sv;
                        st2 += sv * (ep.stat_mode == 1 ? sv : qa * msk[u] + qb);
                    }
                }
            }
        }
        if (ep.stat_mode) {
            // per-column partial sums of this CTA's 128 rows, fixed order: lanes sharing a column, then the 4 lane quarters
#pragma unroll
            for (int o = CW; o < 32; o <<= 1) {
                st1 += __shfl_xor_sync(0xffffffffu, st1, o);
                st2 += __shfl_xor_sync(0xffffffffu, st2, o);
            }
            double *sstat = reinterpret_cast<double *>(smem + STAGE_BYTES);  // second pipeline stage: free as well
            if (rsub == 0) {
                sstat[(quarter * BN + cg * CW + col) * 2 + 0] = st1;
                sstat[(quarter * BN + cg * CW + col) * 2 + 1] = st2;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");
            if ((int)threadIdx.x < BN && n0 + (int)threadIdx.x < N) {
                double a1 = 0.0, a2 = 0.0;
#pragma unroll
                for (int qd = 0; qd < 4; ++qd) {
                    a1 += sstat[(qd * BN + threadIdx.x) * 2 + 0];
                    a2 += sstat[(qd * BN + threadIdx.x) * 2 + 1];
                }
                double *dst = ep.stats + ((long long)blockIdx.y * N + n0 + threadIdx.x) * 2;
                dst[0] = a1, dst[1] = a2;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS)
                     : "memory");
    }
}

// ---- operand slicing ------------------------------------------------------------------------------------------------
constexpr int EXP_SENTINEL = (int)0x80808080;  // cudaMemsetAsync(0x80) pattern: below every real exponent

__device__ __forceinline__ int exponent_above(double amax) {  // smallest e with amax < 2^e (sentinel for amax == 0)
    if (!(amax > 0.0)) return EXP_SENTINEL;
    int e = (int)((__double_as_longlong(amax) >> 52) & 0x7ff) - 1022;
    return e < -960 ? -960 : (e > 960 ? 960 : e);
}
__device__ __forceinline__ int exponent_or_zero(int e) { return e == EXP_SENTINEL ? 0 : e; }

template <typename T>
__device__ __forceinline__ T block_max(T v, T *sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    T r = sh[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = fmax(r, sh[w]);
    __syncthreads();
    return r;
}

__device__ __forceinline__ float tf32_round(float x) {  // round to nearest even on the 10-bit mantissa
    uint32_t u = __float_as_uint(x);
    if ((u & 0x7f800000u) == 0x7f800000u) return x;
    u += 0xfffu + ((u >> 13) & 1u);
    return __uint_as_float(u & 0xffffe000u);
}

// Digits of NV values already scaled by 2^(LEAD - e) (|v| < 2^LEAD), packed little-endian, one signed byte per digit:
// digit_s = rint(v), v <- RADIX (v - digit_s); the remainder after S digits (at most half a unit of the last digit) is
// dropped.  Base 128: digits in [-64, 64].  Base 256 (dense): rint gives [-128, 128]; a digit above 127 is lowered by 256
// with a carry into the next more significant one (the leading digit has a bit to spare), so every digit is a signed byte
// and the digits stay balanced -- products of dropped digit pairs have random signs, no bias.
template <int KIND, int NV>
__device__ __forceinline__ void digits(double (&res)[NV], uint32_t (&pack)[Cfg<KIND>::S][NV / 4]) {
    using C = Cfg<KIND>;
#pragma unroll
    for (int s = 0; s < C::S; ++s)
#pragma unroll
        for (int w = 0; w < NV / 4; ++w) pack[s][w] = 0;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        int d[C::S];
        double r = res[q];
#pragma unroll
        for (int s = 0; s < C::S; ++s) {
            const double qd = rint(r);
            r = (r - qd) * (double)(1 << C::BASE_BITS);
            d[s] = (int)qd;
        }
        if constexpr (C::DENSE) {
#pragma unroll
            for (int s = C::S - 1; s >= 1; --s)
                if (d[s] > 127) d[s] -= 256, d[s - 1] += 1;
        }
#pragma unroll
        for (int s = 0; s < C::S; ++s) pack[s][q >> 2] |= ((uint32_t)d[s] & 0xffu) << (8 * (q & 3));
    }
}

// Row slicing: operand row r = x[r][0..k).  One block per row.  out: [S][rows][pitch bytes].
template <int KIND>
__global__ void slice_rows_kernel(const void *xin, long long ldx, int rows, int k, uint8_t *out, long long pitch,
                                  int *exps) {
    pdl_launch_dependents();
    pdl_wait();
    using C = Cfg<KIND>;
    const int r = blockIdx.x;
    const long long slice_stride = (long long)rows * pitch;
    if constexpr (C::INT) {
        __shared__ double sh[8];
        const double *x = reinterpret_cast<const double *>(xin) + (long long)r * ldx;
        double amax = 0.0;
        for (int c = threadIdx.x; c < k; c += blockDim.x) amax = fmax(amax, fabs(x[c]));
        amax = block_max(amax, sh);
        const int e = exponent_or_zero(exponent_above(amax));
        if (threadIdx.x == 0) exps[r] = e;
        const double sc = pow2(C::LEAD_BITS - e);
        uint8_t *o = out + (long long)r * pitch;
        for (int c = threadIdx.x * 4; c < k; c += blockDim.x * 4) {
            double res[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) res[q] = (c + q < k) ? x[c + q] * sc : 0.0;
            uint32_t pack[C::S][1];
            digits<KIND, 4>(res, pack);
#pragma unroll
            for (int s = 0; s < C::S; ++s)
                *reinterpret_cast<uint32_t *>(o + s * slice_stride + c) = pack[s][0];  // pitch % 128 == 0: in bounds
        }
    } else {
        const float *x = reinterpret_cast<const float *>(xin) + (long long)r * ldx;
        float *o = reinterpret_cast<float *>(out + (long long)r * pitch);
        float *o1 = reinterpret_cast<float *>(out + slice_stride + (long long)r * pitch);
        for (int c = threadIdx.x; c < k; c += blockDim.x) {
            const float v = x[c], hi = tf32_round(v);
            o[c] = hi;
            o1[c] = v - hi;
        }
    }
}

// Column slicing (operand = x^T: operand row c = column c of x, reduction over the rows of x), three small kernels:
//   col_exponent_kernel  per-column exponent: every block takes 32 columns x 256 rows, atomicMax on exps[c] (an integer
//                        maximum: exact and order independent; exps is preset to the sentinel)
//   slice_cols_kernel    32 columns x 128 rows per block: a thread turns 16 consecutive rows of its column into one
//                        16-byte store per slice (fp32: two coalesced-by-row streams through a shared-memory transpose)
//   col_sum_kernel       colsum[c] += coef * sum_r x[r][c] in a fixed order (bias gradients)
__global__ void col_exponent_kernel(const double *x, long long ldx, int rows, int cols, int *exps, double *colsum,
                                    double coef) {
    pdl_launch_dependents();
    pdl_wait();
    const int cl = threadIdx.x & 31, rg = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + cl;
    const int rbeg = blockIdx.y * 256 + rg * 32, rend = min(rows, rbeg + 32);
    __shared__ double sh[8][33], ss[8][33];
    double amax = 0.0, sum = 0.0;
    if (c < cols)
        for (int r = rbeg; r < rend; ++r) {
            const double v = x[(long long)r * ldx + c];
            amax = fmax(amax, fabs(v));
            sum += v;
        }
    sh[rg][cl] = amax;
    ss[rg][cl] = sum;
    __syncthreads();
    if (rg == 0 && c < cols) {
        for (int g = 1; g < 8; ++g) amax = fmax(amax, sh[g][cl]), sum += ss[g][cl];
        const int e = exponent_above(amax);
        if (e != EXP_SENTINEL) atomicMax(exps + c, e);
        if (colsum) colsum[c] += coef * sum;  // only passed when one block covers all rows (fixed summation order)
    }
}

template <int KIND>
__global__ void slice_cols_kernel(const void *xin, long long ldx, int rows, int cols, uint8_t *out, long long pitch,
                                  int *exps) {
    pdl_launch_dependents();
    pdl_wait();
    using C = Cfg<KIND>;
    const long long slice_stride = (long long)cols * pitch;
    if constexpr (C::INT) {
        const int cl = threadIdx.x & 31, rg = threadIdx.x >> 5;
        const int c = blockIdx.x * 32 + cl;
        const int r0 = blockIdx.y * 128 + rg * 16;
        if (c >= cols || r0 >= rows) return;
        const double *x = reinterpret_cast<const double *>(xin);
        const int e = exponent_or_zero(exps[c]);  // blocks with blockIdx.y > 0 may read the sentinel or the 0 written below
        if (blockIdx.y == 0 && rg == 0 && exps[c] == EXP_SENTINEL) exps[c] = 0;
        const double sc = pow2(C::LEAD_BITS - e);
        double res[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) res[q] = (r0 + q < rows) ? x[(long long)(r0 + q) * ldx + c] * sc : 0.0;
        uint32_t pack[C::S][4];
        digits<KIND, 16>(res, pack);
        uint8_t *o = out + (long long)c * pitch + r0;  // r0 % 16 == 0, pitch % 128 == 0: aligned and in bounds
#pragma unroll
        for (int s = 0; s < C::S; ++s)
            *reinterpret_cast<uint4 *>(o + s * slice_stride) = make_uint4(pack[s][0], pack[s][1], pack[s][2], pack[s][3]);
    } else {
        // 32 x 32 transpose tiles: coalesced reads along the columns of x, coalesced writes along its rows
        __shared__ float th[32][33], tl[32][33];
        const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 8 x 32 threads
        const float *x = reinterpret_cast<const float *>(xin);
        const int cbase = blockIdx.x * 32;
        for (int rb = blockIdx.y * 128; rb < min(rows, blockIdx.y * 128 + 128); rb += 32) {
            for (int i = ty; i < 32; i += 8) {
                const int r = rb + i, c = cbase + tx;
                const float v = (r < rows && c < cols) ? x[(long long)r * ldx + c] : 0.f;
                const float hi = tf32_round(v);
                th[i][tx] = hi;
                tl[i][tx] = v - hi;
            }
            __syncthreads();
            for (int i = ty; i < 32; i += 8) {
                const int c = cbase + i, r = rb + tx;
                if (c < cols && r < rows) {
                    reinterpret_cast<float *>(out + (long long)c * pitch)[r] = th[tx][i];
                    reinterpret_cast<float *>(out + slice_stride + (long long)c * pitch)[r] = tl[tx][i];
                }
            }
            __syncthreads();
        }
    }
}

// colsum[c] += coef * sum_r x[r][c], fixed order: 32 columns x 8 row classes (r mod 8) per block.
template <typename T>
__global__ void col_sum_kernel(const T *x, long long ldx, int rows, int cols, T *colsum, double coef) {
    pdl_launch_dependents();
    pdl_wait();
    const int cl = threadIdx.x & 31, rg = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + cl;
    __shared__ double ss[8][33];
    double a0 = 0.0, a1 = 0.0;
    if (c < cols) {
        int r = rg;
        for (; r + 8 < rows; r += 16) {
            a0 += (double)x[(long long)r * ldx + c];
            a1 += (double)x[(long long)(r + 8) * ldx + c];
        }
        if (r < rows) a0 += (double)x[(long long)r * ldx + c];
    }
    ss[rg][cl] = a0 + a1;
    __syncthreads();
    if (rg == 0 && c < cols) {
        double sum = ss[0][cl];
        for (int g = 1; g < 8; ++g) sum += ss[g][cl];
        colsum[c] = (T)((double)colsum[c] + coef * sum);
    }
}

// ---- fused row + column slicing of one source (an activation is the A operand of the next product by rows and the
// B operand of a weight-gradient product by columns): one read of the source per kernel, 32 x 64 tiles --------------------
__global__ void fill_sentinel_kernel(int *a, int na, int *b, int nb) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < na) a[i] = EXP_SENTINEL;
    if (i < nb) b[i] = EXP_SENTINEL;
}

__global__ void exp_both_kernel(const double *x, long long ldx, int rows, int cols, int *exp_r, int *exp_c, double *colpart) {
    pdl_launch_dependents();
    pdl_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c0 = blockIdx.x * 64, r0 = blockIdx.y * 32;
    __shared__ double cm[8][64], cs[8][64];
    double m0 = 0.0, m1 = 0.0, s0 = 0.0, s1 = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = r0 + warp * 4 + i;
        double v0 = 0.0, v1 = 0.0;
        if (r < rows) {
            if (c0 + lane < cols) v0 = x[(long long)r * ldx + c0 + lane];
            if (c0 + lane + 32 < cols) v1 = x[(long long)r * ldx + c0 + lane + 32];
        }
        double rm = fmax(fabs(v0), fabs(v1));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) rm = fmax(rm, __shfl_xor_sync(0xffffffffu, rm, o));
        if (lane == 0 && r < rows) {
            const int e = exponent_above(rm);
            if (e != EXP_SENTINEL) atomicMax(exp_r + r, e);
        }
        m0 = fmax(m0, fabs(v0)), m1 = fmax(m1, fabs(v1));
        s0 += v0, s1 += v1;
    }
    cm[warp][lane] = m0, cm[warp][lane + 32] = m1;
    cs[warp][lane] = s0, cs[warp][lane + 32] = s1;
    __syncthreads();
    if (threadIdx.x < 64 && c0 + (int)threadIdx.x < cols) {
        double m = cm[0][threadIdx.x], sum = cs[0][threadIdx.x];
        for (int w = 1; w < 8; ++w) m = fmax(m, cm[w][threadIdx.x]), sum += cs[w][threadIdx.x];
        const int e = exponent_above(m);
        if (e != EXP_SENTINEL) atomicMax(exp_c + c0 + threadIdx.x, e);
        if (colpart) colpart[(long long)blockIdx.y * cols + c0 + threadIdx.x] = sum;
    }
}

template <int KIND>
__global__ void slice_both_kernel(const double *x, long long ldx, int rows, int cols, uint8_t *out_r, long long pitch_r,
                                  uint8_t *out_c, long long pitch_c, int *exp_r, int *exp_c, double *colsum, double coef,
                                  const double *colpart, int nrt) {
    pdl_launch_dependents();
    pdl_wait();
    using C = Cfg<KIND>;
    __shared__ double tile[32][65];
    const int c0 = blockIdx.x * 64, r0 = blockIdx.y * 32;
    for (int i = threadIdx.x; i < 32 * 64; i += 256) {
        const int r = i >> 6, c = i & 63;
        tile[r][c] = (r0 + r < rows && c0 + c < cols) ? x[(long long)(r0 + r) * ldx + c0 + c] : 0.0;
    }
    __syncthreads();
    // by rows: (row, 4 consecutive columns) -> one 4-byte store per slice
    for (int task = threadIdx.x; task < 512; task += 256) {
        const int r = task >> 4, cg = (task & 15) * 4;
        if (r0 + r < rows && c0 + cg < cols) {
            const double sc = pow2(C::LEAD_BITS - exponent_or_zero(exp_r[r0 + r]));
            double res[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) res[q] = tile[r][cg + q] * sc;
            uint32_t pack[C::S][1];
            digits<KIND, 4>(res, pack);
            uint8_t *o = out_r + (long long)(r0 + r) * pitch_r + c0 + cg;
#pragma unroll
            for (int s = 0; s < C::S; ++s) *reinterpret_cast<uint32_t *>(o + (long long)s * rows * pitch_r) = pack[s][0];
        }
    }
    // by columns: (column, 16 consecutive rows) -> one 16-byte store per slice
    if (threadIdx.x < 128) {
        const int c = threadIdx.x & 63, rg = (threadIdx.x >> 6) * 16;
        if (c0 + c < cols && r0 + rg < rows) {
            const double sc = pow2(C::LEAD_BITS - exponent_or_zero(exp_c[c0 + c]));
            double res[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) res[q] = tile[rg + q][c] * sc;
            uint32_t pack[C::S][4];
            digits<KIND, 16>(res, pack);
            uint8_t *o = out_c + (long long)(c0 + c) * pitch_c + r0 + rg;
#pragma unroll
            for (int s = 0; s < C::S; ++s)
                *reinterpret_cast<uint4 *>(o + (long long)s * cols * pitch_c) = make_uint4(pack[s][0], pack[s][1], pack[s][2], pack[s][3]);
        }
    }
    // all-zero rows / columns keep the sentinel: publish exponent 0 for the products' epilogues (readers treat both alike)
    if (blockIdx.x == 0 && threadIdx.x < 32 && r0 + (int)threadIdx.x < rows && exp_r[r0 + threadIdx.x] == EXP_SENTINEL)
        exp_r[r0 + threadIdx.x] = 0;
    if (blockIdx.y == 0 && threadIdx.x >= 64 && threadIdx.x < 128) {
        const int c = c0 + (int)threadIdx.x - 64;
        if (c < cols) {
            if (exp_c[c] == EXP_SENTINEL) exp_c[c] = 0;
            if (colsum) {
                double sum = 0.0;
                for (int t = 0; t < nrt; ++t) sum += colpart[(long long)t * cols + c];  // fixed order over the row tiles
                colsum[c] += coef * sum;
            }
        }
    }
}

// fp32: hi / lo of every entry in both layouts; column sums of the tile's 32 rows into colpart.
__global__ void slice_both_tf32_kernel(const float *x, long long ldx, int rows, int cols, float *out_r, long long pitch_r,
                                       float *out_c, long long pitch_c, double *colpart) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float th[32][65], tl[32][65];
    const int c0 = blockIdx.x * 64, r0 = blockIdx.y * 32;
    const long long slice_r = (long long)rows * pitch_r, slice_c = (long long)cols * pitch_c;
    for (int i = threadIdx.x; i < 32 * 64; i += 256) {
        const int r = i >> 6, c = i & 63;
        const bool in = r0 + r < rows && c0 + c < cols;
        const float v = in ? x[(long long)(r0 + r) * ldx + c0 + c] : 0.f;
        const float hi = tf32_round(v), lo = v - hi;
        th[r][c] = hi, tl[r][c] = lo;
        if (in) {
            float *o = out_r + (long long)(r0 + r) * pitch_r + c0 + c;
            o[0] = hi, o[slice_r] = lo;
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int c = warp; c < 64; c += 8) {
        if (c0 + c < cols && r0 + lane < rows) {
            float *o = out_c + (long long)(c0 + c) * pitch_c + r0 + lane;
            o[0] = th[lane][c], o[slice_c] = tl[lane][c];
        }
    }
    if (colpart && threadIdx.x < 64 && c0 + (int)threadIdx.x < cols) {
        double sum = 0.0;
        for (int r = 0; r < 32; ++r) sum += (double)th[r][threadIdx.x] + (double)tl[r][threadIdx.x];
        colpart[(long long)blockIdx.y * cols + c0 + threadIdx.x] = sum;
    }
}

__global__ void colsum_finalize_f32_kernel(const double *colpart, int nrt, int cols, float *colsum, double coef) {
    pdl_launch_dependents();
    pdl_wait();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    double sum = 0.0;
    for (int t = 0; t < nrt; ++t) sum += colpart[(long long)t * cols + c];
    colsum[c] = (float)((double)colsum[c] + coef * sum);
}

// ---- host side ------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}


template <int KIND>
static int make_map(CUtensorMap *map, const void *base, int rows, int k, int box_rows) {
    using C = Cfg<KIND>;
    EncodeTiledFn fn = encode_fn();
    PNODE_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
    const long long pitch = pitch_bytes(KIND, k);
    cuuint64_t dims[3] = {(cuuint64_t)k, (cuuint64_t)rows, (cuuint64_t)C::S};
    cuuint64_t strides[2] = {(cuuint64_t)pitch, (cuuint64_t)pitch * (cuuint64_t)rows};
    cuuint32_t box[3] = {(cuuint32_t)(C::KB / C::ELEM), (cuuint32_t)box_rows, 1u};
    cuuint32_t estr[3] = {1u, 1u, 1u};
    CUresult r = fn(map, C::INT ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                    const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    C::KB == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    PNODE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) rows=%d k=%d", (int)r, rows, k);
    return 0;
}

template <int KIND>
static int launch_gemm(const void *a, const void *b, int M, int N, int K, const Epilogue &ep, cudaStream_t stream) {
    using C = Cfg<KIND>;
    constexpr int STAGE_BYTES = C::S * (128 + C::BN) * C::KB;
    constexpr int SMEM = C::STAGES * STAGE_BYTES + 1024 + 256;
    static bool configured = false;
    if (!configured) {
        PNODE_CUDA_OK(cudaFuncSetAttribute(umma_gemm_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        configured = true;
    }
    CUtensorMap ma, mb;
    if (int rc = make_map<KIND>(&ma, a, M, K, 128)) return rc;
    if (int rc = make_map<KIND>(&mb, b, N, K, C::BN)) return rc;
    int splits = 1;
    if (ep.kb_per_split > 0) {
        const int total_kb = (K * C::ELEM + C::KB - 1) / C::KB;
        splits = (total_kb + ep.kb_per_split - 1) / ep.kb_per_split;
    }
    dim3 grid((N + C::BN - 1) / C::BN, (M + 127) / 128, splits);
    PNODE_CUDA_OK(launch_pdl(umma_gemm_kernel<KIND>, dim3(grid), dim3(GEMM_THREADS), SMEM, stream, ma, mb, M, N, K, ep));
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

int gemm_ex(int kind, const void *a, const void *b, int M, int N, int K, const Epilogue &ep, cudaStream_t stream) {
    PNODE_REQUIRE(M > 0 && N > 0 && K > 0 && K <= 65536, "umma gemm: bad shape %d x %d x %d", M, N, K);
    // dense digits: a diagonal accumulates up to S products of 255 x 255 per reduction index in int32
    PNODE_REQUIRE(kind != KIND_I8 || K <= PNODE_I8_MAX_K, "umma gemm: reduction length %d exceeds %d for PNODE_SLICED_I8 "
                  "(use PNODE_SLICED_I8X)", K, PNODE_I8_MAX_K);
    // 8 digit pairs of up to 64 x 64 per reduction index on diagonal 7: 2^31 at K = 65536, one past INT32_MAX
    PNODE_REQUIRE(kind != KIND_I8X || K <= PNODE_I8X_MAX_K, "umma gemm: reduction length %d exceeds %d for PNODE_SLICED_I8X",
                  K, PNODE_I8X_MAX_K);
    if (kind == KIND_I8) return launch_gemm<KIND_I8>(a, b, M, N, K, ep, stream);
    if (kind == KIND_I8X) return launch_gemm<KIND_I8X>(a, b, M, N, K, ep, stream);
    if (kind == KIND_TF32) return launch_gemm<KIND_TF32>(a, b, M, N, K, ep, stream);
    PNODE_REQUIRE(false, "umma gemm: unknown operand kind %d", kind);
}

int gemm(int kind, const void *a, const int *ea, const void *b, const int *eb, int M, int N, int K, void *c,
         long long ldc, double alpha, const void *bias, int relu, const void *mask, long long ldmask, int accumulate,
         cudaStream_t stream) {
    Epilogue ep{};
    ep.C = c, ep.ldc = ldc, ep.ea = ea, ep.eb = eb, ep.alpha = alpha, ep.bias = bias, ep.mask = mask, ep.ldmask = ldmask;
    ep.relu = relu, ep.accumulate = accumulate;
    return gemm_ex(kind, a, b, M, N, K, ep, stream);
}

int split_k_blocks(int kind, int K, int splits) {
    const int kb = kind == KIND_TF32 ? 128 / 4 : 64;
    const int total = (K + kb - 1) / kb;
    return (total + splits - 1) / splits;
}

int slice_rows(int kind, const void *x, long long ldx, int rows, int k, void *out, int *exps, cudaStream_t stream) {
    const long long pitch = pitch_bytes(kind, k);
    if (kind == KIND_I8)
        PNODE_CUDA_OK(launch_pdl(slice_rows_kernel<KIND_I8>, dim3(rows), dim3(256), 0, stream, x, ldx, rows, k, (uint8_t *)out, pitch, exps));
    else if (kind == KIND_I8X)
        PNODE_CUDA_OK(launch_pdl(slice_rows_kernel<KIND_I8X>, dim3(rows), dim3(256), 0, stream, x, ldx, rows, k, (uint8_t *)out, pitch, exps));
    else
        PNODE_CUDA_OK(launch_pdl(slice_rows_kernel<KIND_TF32>, dim3(rows), dim3(256), 0, stream, x, ldx, rows, k, (uint8_t *)out, pitch, exps));
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

int slice_cols(int kind, const void *x, long long ldx, int rows, int cols, void *out, int *exps, void *colsum, double coef,
               cudaStream_t stream) {
    const long long pitch = pitch_bytes(kind, rows);
    dim3 grid((cols + 31) / 32, (rows + 127) / 128);
    if (kind == KIND_TF32) {
        PNODE_CUDA_OK(launch_pdl(slice_cols_kernel<KIND_TF32>, dim3(grid), dim3(256), 0, stream, x, ldx, rows, cols, (uint8_t *)out, pitch, exps));
        if (colsum)
            PNODE_CUDA_OK(launch_pdl(col_sum_kernel<float>, dim3((cols + 31) / 32), dim3(256), 0, stream, (const float *)x, ldx, rows, cols, (float *)colsum, coef));
    } else {
        PNODE_CUDA_OK(cudaMemsetAsync(exps, 0x80, sizeof(int) * (size_t)cols, stream));
        const bool one_chunk = rows <= 256;
        PNODE_CUDA_OK(launch_pdl(col_exponent_kernel, dim3(dim3((cols + 31) / 32, (rows + 255) / 256)), dim3(256), 0, stream, (const double *)x, ldx, rows, cols, exps, one_chunk ? (double *)colsum : nullptr, coef));
        if (kind == KIND_I8)
            PNODE_CUDA_OK(launch_pdl(slice_cols_kernel<KIND_I8>, dim3(grid), dim3(256), 0, stream, x, ldx, rows, cols, (uint8_t *)out, pitch, exps));
        else
            PNODE_CUDA_OK(launch_pdl(slice_cols_kernel<KIND_I8X>, dim3(grid), dim3(256), 0, stream, x, ldx, rows, cols, (uint8_t *)out, pitch, exps));
        if (colsum && !one_chunk)
            PNODE_CUDA_OK(launch_pdl(col_sum_kernel<double>, dim3((cols + 31) / 32), dim3(256), 0, stream, (const double *)x, ldx, rows, cols, (double *)colsum,
                                                                         coef));
    }
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

int slice_both(int kind, const void *x, long long ldx, int rows, int cols, void *out_r, int *exp_r, void *out_c, int *exp_c,
               void *colsum, double coef, double *colpart, cudaStream_t stream) {
    PNODE_REQUIRE(colsum == nullptr || colpart != nullptr, "slice_both: column sums need the partial-sum scratch");
    const long long pitch_r = pitch_bytes(kind, cols), pitch_c = pitch_bytes(kind, rows);
    dim3 grid((cols + 63) / 64, (rows + 31) / 32);
    const int nrt = (int)grid.y;
    if (kind == KIND_TF32) {
        PNODE_CUDA_OK(launch_pdl(slice_both_tf32_kernel, dim3(grid), dim3(256), 0, stream, (const float *)x, ldx, rows, cols, (float *)out_r, pitch_r / 4,
                                                         (float *)out_c, pitch_c / 4, colsum ? colpart : nullptr));
        if (colsum)
            PNODE_CUDA_OK(launch_pdl(colsum_finalize_f32_kernel, dim3((cols + 127) / 128), dim3(128), 0, stream, colpart, nrt, cols, (float *)colsum, coef));
    } else {
        const int n = rows > cols ? rows : cols;
        PNODE_CUDA_OK(launch_pdl(fill_sentinel_kernel, dim3((n + 255) / 256), dim3(256), 0, stream, exp_r, rows, exp_c, cols));
        PNODE_CUDA_OK(launch_pdl(exp_both_kernel, dim3(grid), dim3(256), 0, stream, (const double *)x, ldx, rows, cols, exp_r, exp_c, colsum ? colpart : nullptr));
        if (kind == KIND_I8)
            PNODE_CUDA_OK(launch_pdl(slice_both_kernel<KIND_I8>, dim3(grid), dim3(256), 0, stream, (const double *)x, ldx, rows, cols, (uint8_t *)out_r, pitch_r,
                                                                 (uint8_t *)out_c, pitch_c, exp_r, exp_c, (double *)colsum, coef,
                                                                 colpart, nrt));
        else
            PNODE_CUDA_OK(launch_pdl(slice_both_kernel<KIND_I8X>, dim3(grid), dim3(256), 0, stream, (const double *)x, ldx, rows, cols, (uint8_t *)out_r, pitch_r,
                                                                  (uint8_t *)out_c, pitch_c, exp_r, exp_c, (double *)colsum,
                                                                  coef, colpart, nrt));
    }
    PNODE_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace umma
}  // namespace pnode

using namespace pnode;

extern "C" {

static bool known_kind(int kind) { return kind == PNODE_SLICED_I8 || kind == PNODE_SLICED_TF32 || kind == PNODE_SLICED_I8X; }

int64_t pnode_sliced_bytes(int kind, int rows, int k) {
    if (!known_kind(kind)) return -1;
    return umma::sliced_bytes(kind, rows, k);
}

int pnode_slice_rows(int kind, const void *d_x, int64_t ldx, int rows, int k, void *d_slices, int32_t *d_exp, void *stream) {
    PNODE_REQUIRE(known_kind(kind), "pnode_slice_rows: unknown kind %d", kind);
    PNODE_REQUIRE(rows > 0 && k > 0, "pnode_slice_rows: empty operand");
    return umma::slice_rows(kind, d_x, ldx, rows, k, d_slices, d_exp, (cudaStream_t)stream);
}

int pnode_slice_cols(int kind, const void *d_x, int64_t ldx, int rows, int cols, void *d_slices, int32_t *d_exp,
                     void *d_colsum, double coef, void *stream) {
    PNODE_REQUIRE(known_kind(kind), "pnode_slice_cols: unknown kind %d", kind);
    PNODE_REQUIRE(rows > 0 && cols > 0, "pnode_slice_cols: empty operand");
    return umma::slice_cols(kind, d_x, ldx, rows, cols, d_slices, d_exp, d_colsum, coef, (cudaStream_t)stream);
}

int pnode_sliced_gemm(int kind, const void *d_a, const int32_t *d_a_exp, const void *d_b, const int32_t *d_b_exp, int M,
                      int N, int K, void *d_c, int64_t ldc, double alpha, const void *d_bias, int relu, const void *d_mask,
                      int64_t ldmask, int accumulate, void *stream) {
    return umma::gemm(kind, d_a, d_a_exp, d_b, d_b_exp, M, N, K, d_c, ldc, alpha, d_bias, relu, d_mask, ldmask, accumulate,
                      (cudaStream_t)stream);
}

}  // extern "C"
