// tcgen05 (5th-gen tensor core) int8 implicit GEMM for sm_100a: the hot kernel of the codec.
//
//   D[128 x N] (int32, TMEM)  +=  A[128 x 128B] (smem, gathered rows)  x  W[N x 128B]^T (smem, TMA)
//
// One CTA owns a tile of 128 output rows and up to 256 output channels; the accumulator lives in
// tensor memory for the whole tile, so a sparse convolution is OUTPUT-STATIONARY: all kernel offsets
// that have at least one neighbour in the tile are accumulated by `tcgen05.mma.kind::i8` before a
// single fused epilogue (bias + Q6.25 PReLU + requant [+ residual + PReLU]) writes int8 / Q8.23 once.
// No atomics, no int32 round trip through HBM, deterministic.
//
// Warp roles (192 threads):
//   warps 0-3  gather producers: one output row each; 16-byte cp.async with zero-fill for missing
//              neighbours, written straight into the 128B-swizzled K-major layout the MMA expects;
//              afterwards the same four warps run the epilogue (TMEM lane quarter = warp id).
//   warp 4     weight producer: one TMA box (N x 128 B, SWIZZLE_128B) per pipeline stage.
//   warp 5     TMEM allocation + the single MMA-issuing thread.
// smem stages hand over through mbarriers (full: 128 gather arrivals + TMA transaction bytes; empty:
// tcgen05.commit); the accumulator hands over to the epilogue through one more mbarrier.
//
// Two front-ends share the kernel: MODE_CONV reads the k-major neighbour table of coords.cu, MODE_PAIRS
// reads (in,out) pair lists grouped by weight block (dense linear, occupied-children linear).
//
// Replaces lib/int_sparse_conv/src/gather_gemm_scatter.cu:11-144 / gemm.cu:11-127 (CUTLASS 2.x
// mma.sync m16n8k32, one launch per kernel offset, read-modify-write of D per offset) plus the separate
// element-wise epilogue kernels of src/element_wise/*.cu.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"
#include "epi_nt.cuh"

namespace fpcc {

constexpr int TC_M = 128;         // rows per tile (UMMA M)
constexpr int TC_KB = 128;        // K bytes per stage (one 128B swizzle atom)
constexpr int TC_MAX_KVOL = 32;   // offsets tracked by the per-tile activity mask

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"  // suspend-time hint: sleep in hardware, not in a spin loop
        "@p bra.uni WAIT_DONE;\n\t"
        "bra.uni WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}

// SM100 shared-memory matrix descriptor, K-major, SWIZZLE_128B: 8-row groups are 1024 B apart (SBO),
// the leading-dimension offset is unused for a single 128 B atom along K.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);  // start address, bits [0,14)
    d |= (uint64_t)(1024u >> 4) << 32;             // stride byte offset, bits [32,46)
    d |= (uint64_t)1 << 46;                        // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                        // layout type: SWIZZLE_128B
    return d;
}
// kind::i8 instruction descriptor: D = s32, A = B = s8, both K-major, M = 128, N = n
__device__ __forceinline__ uint32_t umma_idesc_i8(int n) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
}
// kind::f16 instruction descriptor: D = f32, A = B = f16 (fmt 0) or bf16 (fmt 1), K-major, M = 128, N = n
__device__ __forceinline__ uint32_t umma_idesc_f16(int n, int bf16) {
    return (1u << 4) | ((uint32_t)bf16 << 7) | ((uint32_t)bf16 << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------
// kernel
// ---------------------------------------------------------------------------------------------
#ifdef FPCC_TC_TRACE
// Experiment builds only (build.build_variant(name, ['-DFPCC_TC_TRACE'])): CTA 0 writes globaltimer stamps of its roles
// per tile into g_trace[tile_local][slot]; tools/trace_tiles.py reads them back through fpcc_trace_read.
__device__ unsigned long long g_trace[4096][8];
__device__ __forceinline__ void trace_stamp(int j, int slot) {
    if (blockIdx.x == 0 && j < 4096) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_trace[j][slot] = t;
    }
}
#define TRACE(j, slot) trace_stamp((j), (slot))
#else
#define TRACE(j, slot)
#endif

struct TcArgs {
    // common
    const int8_t *A;   // activations [*, K]
    int K;             // contraction bytes (C_in), multiple of 16
    int N;             // output channels of one weight block (C_out)
    int n_tile;        // channels per CTA: multiple of 16, <= 256
    int tmem_cols;     // power of two >= n_tile, >= 32
    // MODE_CONV
    const int32_t *nbr;
    int64_t ld;
    int n_out, kvol;
    const int32_t *row_perm;  // optional: column j of nbr describes output row row_perm[j] (rows grouped by pattern)
    // MODE_PAIRS
    const int32_t *in_idx, *out_idx, *offsets;
    int n_groups, n_pairs, bias_per_group;
};

// ---------------------------------------------------------------------------------------------
// persistent kernel: one CTA per SM loops over tiles; the accumulator is double-buffered in TMEM so the
// epilogue of tile t (8 warps, int64 requant arithmetic) overlaps the gathers + MMAs of tile t+1; TMEM
// allocation, barrier setup and weight-descriptor prefetch are paid once per CTA instead of once per tile.
//
//   warps 0-7   epilogue: TMEM lane quarter = warp % 4, column half = warp / 4
//   warps 8-11  gather producers (one output row per thread) + per-tile metadata (source rows, offset mask)
//   warp 12     weight producer (TMA)          warp 13   TMEM owner + MMA issuer
// ---------------------------------------------------------------------------------------------
// ---------------------------------------------------------------------------------------------
// Integer epilogue.  Two implementations of the reference's arithmetic (bias_prelu_requant.cu:6-37, prelu.cu:6-21,
// cuda_ops.py:82-92):
//   * lean_tile   32-bit registers, ~5 (no PReLU) / ~8.5 (PReLU) instructions per element, taken when the CTA-uniform
//                 and per-channel preconditions proven at staging time hold (every layer of a PTQ-converted model);
//   * epi_chunk   exact 64-bit arithmetic for everything else (odd shifts, huge multipliers, slopes outside [0, 1],
//                 int16 outputs, unaligned rows ...).
// Both give the same integers wherever the lean preconditions hold (tests/test_gpu_ops.py sweeps both).
// ---------------------------------------------------------------------------------------------
constexpr int EC = 16;  // accumulator columns per epilogue step (one tcgen05.ld.32x32b.x16)

// 16-byte vector stores of the packed words of one chunk (nbytes is a multiple of 16)
template <int WORDS>
__device__ __forceinline__ void store_words(char *optr, const uint32_t (&w)[WORDS], int nbytes) {
#pragma unroll
    for (int t = 0; t < WORDS / 4; ++t)
        if (t * 16 < nbytes) reinterpret_cast<uint4 *>(optr)[t] = make_uint4(w[4 * t], w[4 * t + 1], w[4 * t + 2], w[4 * t + 3]);
}

struct EpiCtx {
    const int4 *chan4;         // smem (bias, mul, thr, -) of this chunk
    int32_t slope, post;
    int64_t zp, half;          // half = 2^(shift-1) (0 when shift == 0)
    int shift, sgn;            // sgn = 1 when shift > 0 (round-half-away correction for negatives)
    const int32_t *row_bias;   // entries of the occupancy-indexed bias row of this chunk (ROWBIAS)
    const int32_t *residual;   // entries of this chunk, or NULL
    bool has_post;
    int nvalid;
    int8_t *aux;               // dual output: int8 entries of this chunk, or NULL
};

__device__ __forceinline__ int32_t sat_s8(int64_t r) { int32_t o; asm("cvt.sat.s8.s64 %0, %1;" : "=r"(o) : "l"(r)); return o; }
__device__ __forceinline__ int32_t sat_s16(int64_t r) { int32_t o; asm("cvt.sat.s16.s64 %0, %1;" : "=r"(o) : "l"(r)); return o; }
__device__ __forceinline__ int32_t sat_s32(int64_t r) { int32_t o; asm("cvt.sat.s32.s64 %0, %1;" : "=r"(o) : "l"(r)); return o; }

// exact value of one element before the narrowing store (all 64-bit)
template <int OUT>
__device__ __forceinline__ int32_t epi_exact(int32_t a32, int32_t bias, uint32_t mul, bool has_slope, int32_t slope, int64_t zp,
                                             int64_t half, int sgn, int shift) {
    int64_t v = (int64_t)a32 + (int64_t)bias;
    if (has_slope) {  // Q6.25 PReLU on negatives, round half away (bias_prelu_requant.cu:17-22)
        int64_t t = v * (int64_t)slope;
        t = (t + ((1ll << 24) - (int64_t)((uint64_t)t >> 63))) >> 25;
        v = v < 0 ? t : v;
    }
    int64_t r = v * (int64_t)mul + zp;
    r = (r + (half - (int64_t)(((uint64_t)r >> 63) & (uint64_t)sgn))) >> shift;
    return OUT == FPCC_OUT_I8 ? sat_s8(r) : (OUT == FPCC_OUT_I16 ? sat_s16(r) : sat_s32(r));
}

// Second stage, exact: the consumer's PReLUIn32Out32 (prelu.cu:6-21, saturating) + RequantFxpToScaledInt8
// (requant.cu:7-26) applied to a finished int32 value.
struct Post2 {
    bool on, has_slope;
    bool dual;  // the int32 rows are stored as well (fpcc_epilogue::aux_out); the int8 rows go to the aux pointer
    int32_t slope;
    uint32_t mul;
    int64_t zp;
    int shift;
};
__device__ __forceinline__ Post2 load_post2(const EpiParams &ep) {
    Post2 p2;
    p2.on = ep.post_mul != nullptr;
    p2.dual = p2.on && ep.aux_out != nullptr;
    p2.has_slope = p2.on && ep.post_slope2 != nullptr;
    p2.slope = p2.has_slope ? ep.post_slope2[0] : 0;
    p2.mul = p2.on ? ep.post_mul[0] : 0u;
    p2.zp = p2.on ? ep.post_zp[0] : 0;
    p2.shift = p2.on ? ep.post_shift : 0;
    return p2;
}
__device__ __forceinline__ int32_t post2_exact(int32_t y, const Post2 &p2) {
    int64_t v = (int64_t)y;
    if (p2.has_slope) v = (int64_t)sat_s32(prelu_q25(v, p2.slope));
    return sat_s8(rha_shift(v * (int64_t)p2.mul + p2.zp, p2.shift));
}

template <int OUT, bool SLOPE, bool ROWBIAS>
__device__ __forceinline__ void epi_chunk(const uint32_t (&acc)[EC], const EpiCtx &cx, int32_t (&o)[EC]) {
#pragma unroll
    for (int q = 0; q < EC; ++q) {
        int32_t a32 = (int32_t)acc[q];
        if (ROWBIAS) a32 = (int32_t)((uint32_t)a32 + (uint32_t)__ldg(&cx.row_bias[q < cx.nvalid ? q : 0]));
        o[q] = epi_exact<OUT>(a32, cx.chan4[q].x, (uint32_t)cx.chan4[q].y, SLOPE, cx.slope, cx.zp, cx.half, cx.sgn, cx.shift);
    }
}

// a * b + c in 64 bits, two spellings (measured on B200, profiles/r02_epilogue_variants.txt):
//   mad_wide_c   product pinned to mul.wide.s32, the sum written in C: ptxas picks the instruction from what is USED of the
//                result -- IMAD.HI Rd, Ra, Rb, Rc.64 (high word of the full sum, ONE instruction) where only bits 32..63
//                are consumed (every shift >= 32), IMAD.WIDE with the 64-bit addend as its C operand for the PReLU.
//                int8 linears 0.087 -> 0.083 ms, with PReLU 0.110 -> 0.099 ms, int8 conv 0.198 -> 0.191 ms.
//   mad_wide     inline mad.wide.s32: always IMAD.WIDE + IADD3 + IADD3.X.  Kept where BOTH words of the sum feed a funnel
//                shift (shift < 32, the int32 outputs): there the one-instruction form measured slower (0.141 -> 0.153 ms).
// (With a loop-invariant factor and a plain C product the front end hoists the sign extension and multiplies 64 x 64 bits.)
__device__ __forceinline__ int64_t mad_wide_c(int32_t a, int32_t b, int64_t c) {
    int64_t p;
    asm("mul.wide.s32 %0, %1, %2;" : "=l"(p) : "r"(a), "r"(b));
    return p + c;
}
__device__ __forceinline__ int64_t mad_wide(int32_t a, int32_t b, int64_t c) {
    int64_t d;
    asm("mad.wide.s32 %0, %1, %2, %3;" : "=l"(d) : "r"(a), "r"(b), "l"(c));
    return d;
}
__device__ __forceinline__ int4 lds128(uint32_t addr) {
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
// staged channel constants are written before a barrier and read-only afterwards: a plain (non-volatile) load
__device__ __forceinline__ int4 lds128_ro(uint32_t addr) {
    int4 v;
    asm("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
// 32-byte accesses (sm_100: LDG/STG.E.ENL2.256): one WHOLE sector per lane.  With a row per lane (tcgen05.ld.32x32b) every
// 16-byte store of a row is half a sector; two chunks' worth of an int8 row or 8 columns of an int32 row fill one.
__device__ __forceinline__ void stg256(void *p, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t a4, uint32_t a5, uint32_t a6, uint32_t a7) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(a4), "r"(a5), "r"(a6), "r"(a7) : "memory");
}
__device__ __forceinline__ void ldg256(const void *p, int4 &lo, int4 &hi) {
    asm volatile("ld.global.nc.v8.s32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w) : "l"(p));
}
__device__ __forceinline__ int64_t pack64(uint32_t lo, uint32_t hi) {
    int64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
    return d;
}
// Q6.25 PReLU for 0 <= slope <= 2^25 (|result| <= |v|): rha(v*slope, 25) == (v*slope + 2^24 - 1) >> 25 for v < 0 (the product
// is <= 0 there); for v >= 0 the same expression is <= v, so the PReLU is a plain max.
__device__ __forceinline__ int32_t prelu_unit(int32_t v, int32_t slope, int64_t k24) {
    return max(v, (int32_t)(mad_wide_c(v, slope, k24) >> 25));
}

template <int OUT>
__device__ __forceinline__ void epi_store_chunk(int32_t (&o)[EC], const EpiCtx &cx, void *optr, bool vec, const Post2 &p2) {
    if (OUT == FPCC_OUT_I32 && cx.residual) {
        if (vec) {
            const int4 *rp = reinterpret_cast<const int4 *>(cx.residual);
#pragma unroll
            for (int t = 0; t < EC / 4; ++t) {
                const int4 rv = 4 * t < cx.nvalid ? __ldg(rp + t) : make_int4(0, 0, 0, 0);
                o[4 * t] = (int32_t)((uint32_t)o[4 * t] + (uint32_t)rv.x);  // int32 add wraps
                o[4 * t + 1] = (int32_t)((uint32_t)o[4 * t + 1] + (uint32_t)rv.y);
                o[4 * t + 2] = (int32_t)((uint32_t)o[4 * t + 2] + (uint32_t)rv.z);
                o[4 * t + 3] = (int32_t)((uint32_t)o[4 * t + 3] + (uint32_t)rv.w);
            }
        } else {
#pragma unroll
            for (int q = 0; q < EC; ++q) o[q] = (int32_t)((uint32_t)o[q] + (uint32_t)__ldg(&cx.residual[q < cx.nvalid ? q : 0]));
        }
        if (cx.has_post) {
#pragma unroll
            for (int q = 0; q < EC; ++q) o[q] = sat_s32(prelu_q25((int64_t)o[q], cx.post));
        }
    }
    if (OUT == FPCC_OUT_I32 && p2.on && p2.dual) {  // dual output: int8 rows of the second stage to the aux buffer, int32 rows below
#pragma unroll
        for (int q = 0; q < EC; ++q)
            if (q < cx.nvalid) cx.aux[q] = (int8_t)post2_exact(o[q], p2);
    } else if (OUT == FPCC_OUT_I32 && p2.on) {  // the int32 result feeds the fused second stage; int8 rows are stored
#pragma unroll
        for (int q = 0; q < EC; ++q) o[q] = post2_exact(o[q], p2);
    }
    if (vec) {  // nvalid == EC here (N is a multiple of 16)
        if (OUT == FPCC_OUT_I8 || (OUT == FPCC_OUT_I32 && p2.on && !p2.dual)) {
            uint32_t w[EC / 4];
#pragma unroll
            for (int t = 0; t < EC / 4; ++t) {
                const int q = t * 4;
                uint32_t up;  // saturating pack: d = c[15:0] << 16 | sat8(a) << 8 | sat8(b)
                asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(up) : "r"(o[q + 3]), "r"(o[q + 2]), "r"(0));
                asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(w[t]) : "r"(o[q + 1]), "r"(o[q]), "r"(up));
            }
            store_words<EC / 4>((char *)optr, w, cx.nvalid);
        } else if (OUT == FPCC_OUT_I16) {
            uint32_t w[EC / 2];
#pragma unroll
            for (int t = 0; t < EC / 2; ++t) w[t] = (uint32_t)(o[2 * t] & 0xffff) | ((uint32_t)o[2 * t + 1] << 16);
            store_words<EC / 2>((char *)optr, w, cx.nvalid * 2);
        } else {
            uint32_t w[EC];
#pragma unroll
            for (int t = 0; t < EC; ++t) w[t] = (uint32_t)o[t];
            store_words<EC>((char *)optr, w, cx.nvalid * 4);
        }
    } else {
#pragma unroll
        for (int q = 0; q < EC; ++q) {
            if (q < cx.nvalid) {
                if (OUT == FPCC_OUT_I8 || (OUT == FPCC_OUT_I32 && p2.on && !p2.dual)) ((int8_t *)optr)[q] = (int8_t)max(min(o[q], 127), -128);
                else if (OUT == FPCC_OUT_I16) ((int16_t *)optr)[q] = (int16_t)o[q];
                else ((int32_t *)optr)[q] = o[q];
            }
        }
    }
}

template <int OUT>
__device__ __forceinline__ void epi_dispatch(const uint32_t (&acc)[EC], const EpiCtx &cx, void *optr, bool vec, bool slope, bool rb,
                                             const Post2 &p2) {
    int32_t o[EC];
    if (slope) {
        if (rb) epi_chunk<OUT, true, true>(acc, cx, o);
        else epi_chunk<OUT, true, false>(acc, cx, o);
    } else {
        if (rb) epi_chunk<OUT, false, true>(acc, cx, o);
        else epi_chunk<OUT, false, false>(acc, cx, o);
    }
    epi_store_chunk<OUT>(o, cx, optr, vec, p2);
}

// ---- lean path --------------------------------------------------------------------------------------------------
// t' = v*mul + c0 - [v*mul + zp < 0],  c0 = zp + 2^(shift-1),  result = t' >> shift  (one IMAD.WIDE + one shift).
// How the "-1 for negatives" reaches the 64-bit addend depends on the CTA-uniform case (sign mode):
//   SGN_LO0     zp == 0, shift <= 32: c0 = 2^(shift-1) fits the low word and is >= 1, so c0 - 1 never borrows:
//               lo = c0_lo + (v >> 31) (one LEA.HI.SX32), hi = 0.
//   SGN_HI0     zp == 0, shift >= 33: c0_lo == 0:  lo = sx, hi = c0_hi + sx  with sx = v >> 31.
//   SGN_THR_*   zp != 0 (asymmetric activations feeding a Linear): the sign of v*mul + zp is v < thr[c] with the staged
//               per-channel threshold ceil(-zp / mul); c0_lo != 0 is required so that c0 - 1 stays in the low word.
// *_LO: shift <= 32 (clamped funnel shift of the pair), *_HI: shift >= 32 (arithmetic shift of the high word).
// The accumulator bound |acc| <= K*kvol*127*128 is static, |bias| <= 2^29 and the row-bias bound are checked, so v and
// v*mul + c0 stay inside int32 / int64; a per-channel check proves that the shifted value fits 32 bits for int8 outputs;
// int32 outputs with shift < 32 test the high word per element and redo a chunk exactly when one value saturates.
enum { SGN_LO0 = 0, SGN_HI0 = 1, SGN_THR_LO = 2, SGN_THR_HI = 3, SGN_NONE = -1 };

struct LeanU {
    int32_t slope, post;
    uint32_t c0_lo, c0_hi;
    int shift;
    uint32_t ovf_add, ovf_lim;   // I32, shift < 32: the result fits iff (hi + ovf_add) <= ovf_lim (unsigned)
    uint32_t post2_addr;         // shared-space address of the staged second-stage constants (POST2 instantiations only):
                                 // words {mul2, thr2, slope2, shift2 - 32, c02 lo, c02 hi, nt2},  c02 = zp2 + 2^(shift2 - 1),
                                 // nt2 = 1 when the second stage cannot tie for any int32 input (no sign handling)
    int64_t k24;                 // 2^24 - 1, read back from shared memory: ptxas splits an immediate or uniform 64-bit addend of
                                 // IMAD.WIDE into IADD3 + IMAD.X; a vector register pair stays the instruction's C operand
};

__device__ __forceinline__ int lean_mode(const EpiParams &ep, int64_t zp, int64_t kk, int32_t rb_bound, int64_t *vmax_out) {
    const int shift = ep.shift;
    if (ep.out_type != FPCC_OUT_I8 && ep.out_type != FPCC_OUT_I32) return SGN_NONE;
    if (shift < 1 || shift > 62) return SGN_NONE;
    if (ep.slope) { const int32_t sl = ep.slope[0]; if (sl < 0 || sl > (1 << 25)) return SGN_NONE; }
    if (ep.post_slope) { const int32_t sl = ep.post_slope[0]; if (sl < 0 || sl > (1 << 25)) return SGN_NONE; }
    if (ep.row_bias && (rb_bound <= 0 || ((uintptr_t)ep.row_bias & 15) != 0)) return SGN_NONE;
    if (ep.residual && ((uintptr_t)ep.residual & 15) != 0) return SGN_NONE;
    const int64_t vmax = kk * 16256 + ((int64_t)1 << 29) + (ep.row_bias ? (int64_t)rb_bound : 0);
    if (vmax > 2147483646ll) return SGN_NONE;
    *vmax_out = vmax;
    if (ep.post_mul) {  // fused second stage: int32 first stage in a *_LO mode, shift2 >= 32, threshold representable
        if (ep.out_type != FPCC_OUT_I32 || shift >= 32) return SGN_NONE;
        const uint32_t m2 = ep.post_mul[0];
        const int64_t z2 = ep.post_zp[0];
        if (ep.post_shift < 32 || ep.post_shift > 62 || m2 == 0u || m2 >= (1u << 31) || z2 > ((int64_t)1 << 60) || z2 < -((int64_t)1 << 60)) return SGN_NONE;
        if (ep.post_slope2) { const int32_t sl = ep.post_slope2[0]; if (sl < 0 || sl > (1 << 25)) return SGN_NONE; }
        const int64_t nz = -z2, m = (int64_t)m2, t2 = nz >= 0 ? (nz + m - 1) / m : -((-nz) / m);
        if (t2 > 2147483647ll) return SGN_NONE;  // y == INT32_MAX must still compare right
    }
    if (zp == 0) return shift <= 32 ? SGN_LO0 : SGN_HI0;
    if (zp > ((int64_t)1 << 60) || zp < -((int64_t)1 << 60)) return SGN_NONE;
    const int64_t c0 = zp + ((int64_t)1 << (shift - 1));
    if ((uint32_t)c0 == 0u) return SGN_NONE;
    return shift < 32 ? SGN_THR_LO : SGN_THR_HI;
}

// Stages (bias, mul, thr) of one channel; returns false when the channel cannot take the lean path.
__device__ __forceinline__ bool stage_channel(int32_t bias, uint32_t mul, int64_t zp, int shift, int out_type, int64_t vmax, int4 *ch) {
    bool ok = mul < (1u << 31) && bias <= (1 << 29) && bias >= -(1 << 29);
    if (out_type == FPCC_OUT_I8 || shift >= 32) {  // the shifted value must fit 32 bits (int32 outputs with shift < 32 test per element)
        const int64_t azp = zp < 0 ? -zp : zp;
        const int64_t top = vmax * (int64_t)(mul & 0x7fffffffu) + azp + ((int64_t)1 << (shift - (shift > 0)));
        ok = ok && (top >> shift) < 2147483647ll;
    }
    int64_t t;
    if (mul == 0) t = zp < 0 ? 2147483647ll : -2147483648ll;
    else { const int64_t nz = -zp, m = (int64_t)mul; t = nz >= 0 ? (nz + m - 1) / m : -((-nz) / m); }
    t = t > 2147483647ll ? 2147483647ll : (t < -2147483648ll ? -2147483648ll : t);
    *ch = make_int4(bias, (int32_t)mul, (int32_t)t, 0);
    return ok;
}

// The first stage has ONE sign-exact body.  A second, tie-free body per 16-channel chunk (no sign handling where no channel
// of the chunk can tie, epi_nt.cuh) was measured slower on B200: int8 linear 0.083 -> 0.096 ms from code size and spills at
// the 80-register cap (profiles/r02_epilogue_variants.txt).  The fused second stage uses the tie analysis (one CTA-uniform
// test, no extra body per chunk).
template <int OUT, bool SLOPE, int SGN>
__device__ __forceinline__ bool lean_chunk(const uint32_t (&acc)[EC], uint32_t chan_addr, const LeanU &u, int32_t (&o)[EC]) {
    bool bad = false;
#pragma unroll
    for (int q = 0; q < EC; ++q) {
        const int4 ch = lds128(chan_addr + q * 16);
        int32_t v = (int32_t)acc[q] + ch.x;
        if (SLOPE) v = prelu_unit(v, u.slope, u.k24);
        int64_t add;
        if (SGN == SGN_LO0) {
            add = (int64_t)(uint64_t)(u.c0_lo + (uint32_t)(v >> 31));
        } else if (SGN == SGN_HI0) {
            const uint32_t sx = (uint32_t)(v >> 31);
            add = pack64(sx, u.c0_hi + sx);
        } else {
            add = pack64(v < ch.z ? u.c0_lo - 1u : u.c0_lo, u.c0_hi);
        }
        const int64_t t = (SGN == SGN_HI0 || SGN == SGN_THR_HI) ? mad_wide_c(v, ch.y, add) : mad_wide(v, ch.y, add);
        const uint32_t lo = (uint32_t)t, hi = (uint32_t)((uint64_t)t >> 32);
        int32_t r;
        if (SGN == SGN_LO0 || SGN == SGN_THR_LO) {
            r = (int32_t)__funnelshift_rc(lo, hi, u.shift);
            if (OUT == FPCC_OUT_I32) bad |= hi + u.ovf_add > u.ovf_lim;
        } else {
            r = (int32_t)hi >> (u.shift - 32);
        }
        o[q] = r;  // I8: saturated by the packing conversion
    }
    return !bad;
}

struct LeanTile {
    uint32_t tacc;              // TMEM address of this warp's lane quarter, column 0 of the tile
    uint32_t chan_addr;         // shared-space address of the staged channel constants of column 0
    int c_begin, c_end, ncols;  // this warp's columns; valid columns of the tile (N - n0)
    int n0, ncols_total;        // first channel of the tile, N
    bool have_acc, row_ok;
    char *orow;                 // output row (column n0), NULL rows are not stored
    const int32_t *rb_row;      // occupancy bias row (column n0) or NULL
    const int32_t *res_row;     // residual row (column n0) or NULL
    bool has_post;
    int8_t *aux_row;            // dual output: int8 row (column n0) of fpcc_epilogue::aux_out, or NULL
    bool al32;                  // 256-bit stores allowed: conv kernel (96 registers) and a 32-byte aligned output base.  The
                                // linear kernels sit at their 80-register cap: holding 16 bytes across a chunk costs them 5-20 %
};

__device__ __forceinline__ void tmem_ld1(uint32_t taddr, uint32_t &r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Exact recomputation of one chunk, one column at a time straight from TMEM (rare: an int32 output saturated).
// Executed by the whole warp (tcgen05.ld is warp-collective); rows without an output skip the store.
template <int OUT, bool SLOPE>
__device__ __forceinline__ void lean_redo_chunk(const LeanTile &lt, const LeanU &u, int c0, int64_t zp, const EpiParams &ep) {
    const int64_t half = (int64_t)1 << (u.shift - 1);
    const Post2 p2 = load_post2(ep);
#pragma unroll 1
    for (int q = 0; q < EC; ++q) {
        uint32_t a = 0;
        __syncwarp();  // tcgen05.ld is .sync.aligned: the lanes that skipped the previous column's store rejoin here
        if (lt.have_acc) tmem_ld1(lt.tacc + (uint32_t)(c0 + q), a);
        if (lt.row_ok) {
            const int4 ch = lds128(lt.chan_addr + (uint32_t)(c0 + q) * 16);
            int32_t a32 = (int32_t)a;
            if (lt.rb_row) a32 = (int32_t)((uint32_t)a32 + (uint32_t)__ldg(lt.rb_row + c0 + q));
            int32_t r = epi_exact<OUT>(a32, ch.x, (uint32_t)ch.y, SLOPE, u.slope, zp, half, 1, u.shift);
            if (OUT == FPCC_OUT_I32) {
                if (lt.res_row) {
                    r = (int32_t)((uint32_t)r + (uint32_t)__ldg(lt.res_row + c0 + q));
                    if (lt.has_post) r = sat_s32(prelu_q25((int64_t)r, u.post));
                }
                if (p2.on && lt.aux_row) {  // dual output
                    ((int32_t *)lt.orow)[c0 + q] = r;
                    lt.aux_row[c0 + q] = (int8_t)post2_exact(r, p2);
                } else if (p2.on) {
                    ((int8_t *)lt.orow)[c0 + q] = (int8_t)post2_exact(r, p2);
                } else {
                    ((int32_t *)lt.orow)[c0 + q] = r;
                }
            } else {
                ((int8_t *)lt.orow)[c0 + q] = (int8_t)r;
            }
        }
    }
    __syncwarp();
}

// All chunks of one tile row.  The case (output type, PReLU, sign mode) is chosen once per tile by the caller; row
// pointers and constants are formed once.  Requires 16-byte aligned rows and N % 16 == 0 (whole chunks).
// POST2 (int32 first stage only): the int32 values go through the fused second stage ([PReLU] + requant, shift2 >= 32)
// and leave as int8 rows: y*mul2 + c02 - [y < thr2], high word >> (shift2 - 32).
template <int OUT, bool SLOPE, int SGN, bool POST2, bool SLOPE2, bool RESPF>
__device__ __forceinline__ void lean_tile(const LeanTile &lt, const LeanU &u, int64_t zp, const EpiParams &ep) {
    constexpr int esz = (OUT == FPCC_OUT_I8 || POST2) ? 1 : 4;
    // int32 residual rows (ResBlock conv2) come from HBM: the loads of chunk c+1 are issued before the arithmetic of
    // chunk c (one register set ahead), so that their latency hides behind it instead of stalling every chunk
    // (RESPF: the conv kernel only; the linear kernel sits at its 80-register cap and has no residual user)
    const bool res_on = RESPF && OUT == FPCC_OUT_I32 && lt.res_row != nullptr && lt.row_ok;
    const int c_last = min(lt.c_end, lt.ncols);
    int4 rnext[EC / 4];
#pragma unroll
    for (int t = 0; t < EC / 4; ++t) rnext[t] = make_int4(0, 0, 0, 0);
    if (res_on && lt.c_begin < c_last) {
#pragma unroll
        for (int t = 0; t < EC / 4; ++t) rnext[t] = __ldg(reinterpret_cast<const int4 *>(lt.res_row + lt.c_begin) + t);
    }
    // 32-byte stores need 32-byte aligned pieces: the warp's first column and the row pitch are multiples of 32 bytes
    const bool wide8 = esz == 1 && (lt.c_begin & 31) == 0 && (lt.ncols_total & 31) == 0 && (lt.n0 & 31) == 0 && lt.al32;
    const bool wide32 = esz == 4 && (lt.ncols_total & 7) == 0 && lt.al32;
    uint32_t held[4] = {0u, 0u, 0u, 0u};
    bool held_valid = false;  // per lane: the even chunk of a pair waits for its odd neighbour
    for (int c0 = lt.c_begin; c0 < lt.c_end; c0 += EC) {
        uint32_t acc[EC];
        int4 rcur[EC / 4];
#pragma unroll
        for (int t = 0; t < EC / 4; ++t) rcur[t] = rnext[t];
        if (res_on && c0 + EC < c_last) {
#pragma unroll
            for (int t = 0; t < EC / 4; ++t) rnext[t] = __ldg(reinterpret_cast<const int4 *>(lt.res_row + c0 + EC) + t);
        }
        __syncwarp();  // lanes without an output row skipped the previous chunk's stores
        if (lt.have_acc) {
            tmem_ld16(lt.tacc + (uint32_t)c0, acc);  // .sync.aligned: every lane, also those without a row
        } else {
#pragma unroll
            for (int q = 0; q < EC; ++q) acc[q] = 0;
        }
        if (c0 >= lt.ncols) continue;  // warp-uniform
        if (lt.rb_row) {               // warp-uniform; every lane has its own table row
            const int4 *rp = reinterpret_cast<const int4 *>(lt.rb_row + c0);
#pragma unroll
            for (int t = 0; t < EC / 4; ++t) {
                const int4 rv = lt.row_ok ? __ldg(rp + t) : make_int4(0, 0, 0, 0);
                acc[4 * t] += (uint32_t)rv.x; acc[4 * t + 1] += (uint32_t)rv.y; acc[4 * t + 2] += (uint32_t)rv.z; acc[4 * t + 3] += (uint32_t)rv.w;
            }
        }
        int32_t o[EC];
        const bool good = lean_chunk<OUT, SLOPE, SGN>(acc, lt.chan_addr + (uint32_t)c0 * 16, u, o);
        if (OUT == FPCC_OUT_I32 && (SGN == SGN_LO0 || SGN == SGN_THR_LO)) {
            if (__any_sync(0xffffffffu, !good)) {  // warp-uniform, rare
                if (held_valid) {  // the redo stores this chunk itself: flush the waiting even chunk of the pair first
                    *reinterpret_cast<uint4 *>(lt.orow + (size_t)(c0 - EC) * esz) = make_uint4(held[0], held[1], held[2], held[3]);
                    held_valid = false;
                }
                lean_redo_chunk<OUT, SLOPE>(lt, u, c0, zp, ep);
                continue;
            }
        }
        if (!lt.row_ok) continue;
        if (OUT == FPCC_OUT_I32) {
            if (lt.res_row) {
#pragma unroll
                for (int t = 0; t < EC / 4; ++t) {
                    const int4 rv = RESPF ? rcur[t] : __ldg(reinterpret_cast<const int4 *>(lt.res_row + c0) + t);
                    o[4 * t] = (int32_t)((uint32_t)o[4 * t] + (uint32_t)rv.x);  // int32 add wraps
                    o[4 * t + 1] = (int32_t)((uint32_t)o[4 * t + 1] + (uint32_t)rv.y);
                    o[4 * t + 2] = (int32_t)((uint32_t)o[4 * t + 2] + (uint32_t)rv.z);
                    o[4 * t + 3] = (int32_t)((uint32_t)o[4 * t + 3] + (uint32_t)rv.w);
                }
                if (lt.has_post) {
#pragma unroll
                    for (int q = 0; q < EC; ++q) o[q] = prelu_unit(o[q], u.post, u.k24);
                }
            }
            if (POST2) {
                const int4 k2 = lds128(u.post2_addr);          // mul2, thr2, slope2, shift2 - 32
                const int4 k3 = lds128(u.post2_addr + 16);     // c02 lo, c02 hi, nt2
                const int64_t c02 = pack64((uint32_t)k3.x, (uint32_t)k3.y), c02m1 = c02 - 1;
                if (k3.z) {  // CTA-uniform: no int32 input can tie in the second stage, no sign handling
#pragma unroll
                    for (int q = 0; q < EC; ++q) {
                        int32_t y = o[q];
                        if (SLOPE2) y = prelu_unit(y, k2.z, u.k24);
                        const int64_t t2 = mad_wide_c(y, k2.x, c02);
                        o[q] = (int32_t)((uint64_t)t2 >> 32) >> k2.w;
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < EC; ++q) {
                        int32_t y = o[q];
                        if (SLOPE2) y = prelu_unit(y, k2.z, u.k24);
                        const int64_t t2 = mad_wide_c(y, k2.x, y < k2.y ? c02m1 : c02);
                        o[q] = (int32_t)((uint64_t)t2 >> 32) >> k2.w;
                    }
                }
            } else {
                if (wide32) {  // 64 bytes of the int32 row: two whole sectors
                    char *op = lt.orow + (size_t)c0 * esz;
                    stg256(op, o[0], o[1], o[2], o[3], o[4], o[5], o[6], o[7]);
                    stg256(op + 32, o[8], o[9], o[10], o[11], o[12], o[13], o[14], o[15]);
                } else {
                    uint4 *op = reinterpret_cast<uint4 *>(lt.orow + (size_t)c0 * esz);
#pragma unroll
                    for (int t = 0; t < EC / 4; ++t) op[t] = make_uint4((uint32_t)o[4 * t], (uint32_t)o[4 * t + 1], (uint32_t)o[4 * t + 2], (uint32_t)o[4 * t + 3]);
                }
            }
        }
        if (OUT == FPCC_OUT_I32 && !POST2) {
            // stored above
        } else {
            uint32_t w[EC / 4];
#pragma unroll
            for (int t = 0; t < EC / 4; ++t) {
                const int q = t * 4;
                uint32_t up;  // saturating pack: d = c[15:0] << 16 | sat8(a) << 8 | sat8(b)
                asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(up) : "r"(o[q + 3]), "r"(o[q + 2]), "r"(0));
                asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(w[t]) : "r"(o[q + 1]), "r"(o[q]), "r"(up));
            }
            if (wide8) {
                // even chunk of a pair: hold its 16 bytes; odd chunk: one 32-byte store of both (a whole sector per lane)
                if ((((c0 - lt.c_begin) >> 4) & 1) == 0 && c0 + EC < c_last) {
                    held[0] = w[0]; held[1] = w[1]; held[2] = w[2]; held[3] = w[3];
                    held_valid = true;
                } else if (held_valid) {
                    stg256(lt.orow + (size_t)(c0 - EC) * esz, held[0], held[1], held[2], held[3], w[0], w[1], w[2], w[3]);
                    held_valid = false;
                } else {
                    *reinterpret_cast<uint4 *>(lt.orow + (size_t)c0 * esz) = make_uint4(w[0], w[1], w[2], w[3]);
                }
            } else {
                *reinterpret_cast<uint4 *>(lt.orow + (size_t)c0 * esz) = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
    }
}

template <int OUT, bool SLOPE, bool POST2, bool SLOPE2, bool RESPF>
__device__ __forceinline__ void lean_tile_sgn(const LeanTile &lt, const LeanU &u, int64_t zp, int sgn, const EpiParams &ep) {
    if (POST2) {  // int32 producers of a converted model sit at shift - 23 = 5..16: the *_LO modes
        if (sgn == SGN_LO0) lean_tile<OUT, SLOPE, SGN_LO0, POST2, SLOPE2, RESPF>(lt, u, zp, ep);
        else lean_tile<OUT, SLOPE, SGN_THR_LO, POST2, SLOPE2, RESPF>(lt, u, zp, ep);
        return;
    }
    if (sgn == SGN_HI0) lean_tile<OUT, SLOPE, SGN_HI0, false, false, RESPF>(lt, u, zp, ep);
    else if (sgn == SGN_LO0) lean_tile<OUT, SLOPE, SGN_LO0, false, false, RESPF>(lt, u, zp, ep);
    else if (sgn == SGN_THR_HI) lean_tile<OUT, SLOPE, SGN_THR_HI, false, false, RESPF>(lt, u, zp, ep);
    else lean_tile<OUT, SLOPE, SGN_THR_LO, false, false, RESPF>(lt, u, zp, ep);
}

// ---- quad layout for int32 outputs ------------------------------------------------------------------------------------
// Row-per-lane (tcgen05.ld.32x32b) makes every global access of an int32 row a 16-byte piece in its own sector: a
// STG.128 / LDG.128 touches 32 lines (32 L1 wavefronts) and writes HALF sectors (SM->L2 write bytes = 2x the output;
// measured on the ResBlock conv2 and the logits linears).  tcgen05.ld.16x256b hands the accumulator out so that the four
// lanes of a quad hold 8 consecutive columns of ONE row: lane 4i+j gets columns 2j, 2j+1 (and +8 with .x2) of rows i and
// i+8.  An 8-byte access per lane then covers whole 32-byte sectors per quad, 8 lines per instruction.
__device__ __forceinline__ void tmem_ld_q16(uint32_t taddr, uint32_t (&r)[16]) {  // 32 rows x 16 columns: two 16x256b.x2 loads
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr));
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr + (16u << 16)));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

struct QuadRows {
    int64_t off[4];        // element offset (row * N + n0) of rows q, q+8, q+16, q+24 of this warp's quarter, -1 = no row
    int32_t rb[4];         // row of the occupancy bias table for each of them
};

// register r of tmem_ld_q16 -> (row slot 0..3, channel slot 0..3): rows {q, q+8 | q+16, q+24}, channels {2j, 2j+1, 8+2j, 9+2j}
__device__ __forceinline__ constexpr int quad_row(int r) { return (r >> 3) * 2 + ((r >> 1) & 1); }
__device__ __forceinline__ constexpr int quad_chn(int r) { return ((r >> 2) & 1) * 2 + (r & 1); }

template <bool SLOPE, int SGN, bool RESPF>
__device__ __forceinline__ void quad_tile(const LeanTile &lt, const QuadRows &qr, const LeanU &u, int64_t zp, const EpiParams &ep,
                                          int32_t *out) {
    const int j2 = (threadIdx.x & 3) * 2;
    const int c_last = min(lt.c_end, lt.ncols);
    const bool res_pf = RESPF && ep.residual != nullptr;
    int2 rnext[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) rnext[t] = make_int2(0, 0);
    auto load_res = [&](int c0, int2 (&dst)[8]) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int b = 0; b < 2; ++b)
                dst[i * 2 + b] = qr.off[i] >= 0 ? __ldg(reinterpret_cast<const int2 *>(ep.residual + qr.off[i] + c0 + 8 * b + j2)) : make_int2(0, 0);
    };
    if (res_pf && lt.c_begin < c_last) load_res(lt.c_begin, rnext);
    for (int c0 = lt.c_begin; c0 < lt.c_end; c0 += EC) {
        uint32_t acc[16];
        int2 rcur[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) rcur[t] = rnext[t];
        if (res_pf && c0 + EC < c_last) load_res(c0 + EC, rnext);
        __syncwarp();
        tmem_ld_q16(lt.tacc + (uint32_t)c0, acc);
        if (c0 >= lt.ncols) continue;  // warp-uniform
        if (ep.row_bias) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    const int2 rv = qr.off[i] >= 0 ? __ldg(reinterpret_cast<const int2 *>(ep.row_bias + (int64_t)qr.rb[i] * (lt.ncols_total) + lt.n0 + c0 + 8 * b + j2))
                                                   : make_int2(0, 0);
                    const int r0 = (i >> 1) * 8 + b * 4 + (i & 1) * 2;
                    acc[r0] += (uint32_t)rv.x; acc[r0 + 1] += (uint32_t)rv.y;
                }
        }
        int4 ch[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) ch[k] = lds128_ro(lt.chan_addr + (uint32_t)(c0 + (k >> 1) * 8 + j2 + (k & 1)) * 16);
        int32_t o[16];
        bool bad = false;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const int4 c = ch[quad_chn(r)];
            int32_t v = (int32_t)acc[r] + c.x;
            if (SLOPE) v = prelu_unit(v, u.slope, u.k24);
            int64_t add;
            if (SGN == SGN_LO0) {
                add = (int64_t)(uint64_t)(u.c0_lo + (uint32_t)(v >> 31));
            } else if (SGN == SGN_HI0) {
                const uint32_t sx = (uint32_t)(v >> 31);
                add = pack64(sx, u.c0_hi + sx);
            } else {
                add = pack64(v < c.z ? u.c0_lo - 1u : u.c0_lo, u.c0_hi);
            }
            const int64_t t = (SGN == SGN_HI0 || SGN == SGN_THR_HI) ? mad_wide_c(v, c.y, add) : mad_wide(v, c.y, add);
            const uint32_t lo = (uint32_t)t, hi = (uint32_t)((uint64_t)t >> 32);
            if (SGN == SGN_LO0 || SGN == SGN_THR_LO) {
                o[r] = (int32_t)__funnelshift_rc(lo, hi, u.shift);
                bad |= hi + u.ovf_add > u.ovf_lim;
            } else {
                o[r] = (int32_t)hi >> (u.shift - 32);
            }
        }
        if (SGN == SGN_LO0 || SGN == SGN_THR_LO) {
            if (__any_sync(0xffffffffu, bad)) {  // warp-uniform, rare: exact per-column redo in the row-per-lane layout
                lean_redo_chunk<FPCC_OUT_I32, SLOPE>(lt, u, c0, zp, ep);
                continue;
            }
        }
        if (ep.residual) {
            int2 rr[8];
            if (res_pf) {
#pragma unroll
                for (int t = 0; t < 8; ++t) rr[t] = rcur[t];
            } else {
                load_res(c0, rr);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    const int r0 = (i >> 1) * 8 + b * 4 + (i & 1) * 2;
                    o[r0] = (int32_t)((uint32_t)o[r0] + (uint32_t)rr[i * 2 + b].x);  // int32 add wraps
                    o[r0 + 1] = (int32_t)((uint32_t)o[r0 + 1] + (uint32_t)rr[i * 2 + b].y);
                }
            if (lt.has_post) {
#pragma unroll
                for (int r = 0; r < 16; ++r) o[r] = prelu_unit(o[r], u.post, u.k24);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                const int r0 = (i >> 1) * 8 + b * 4 + (i & 1) * 2;
                if (qr.off[i] >= 0) *reinterpret_cast<int2 *>(out + qr.off[i] + c0 + 8 * b + j2) = make_int2(o[r0], o[r0 + 1]);
            }
        if (ep.aux_out) {
            // dual output (kernel-uniform): the consumer's [PReLU +] requant of the finished int32 values, stored as int8 rows
            // beside them -- y*mul2 + c02 - [y < thr2] (no sign handling when the tie analysis allows), high word >> (shift2 - 32)
            const int4 k2 = lds128(u.post2_addr);       // mul2, thr2, slope2, shift2 - 32
            const int4 k3 = lds128(u.post2_addr + 16);  // c02 lo, c02 hi, nt2
            const int64_t c02 = pack64((uint32_t)k3.x, (uint32_t)k3.y), c02m1 = c02 - 1;
            const bool s2 = ep.post_slope2 != nullptr, nt2 = k3.z != 0;
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                int32_t y = o[r];
                if (s2) y = prelu_unit(y, k2.z, u.k24);
                const int64_t t2 = mad_wide_c(y, k2.x, (nt2 || y >= k2.y) ? c02 : c02m1);
                o[r] = (int32_t)((uint64_t)t2 >> 32) >> k2.w;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    const int r0 = (i >> 1) * 8 + b * 4 + (i & 1) * 2;
                    uint32_t w;  // sat8(o[r0 + 1]) << 8 | sat8(o[r0])
                    asm("cvt.pack.sat.s8.s32.b32 %0, %1, %2, %3;" : "=r"(w) : "r"(o[r0 + 1]), "r"(o[r0]), "r"(0));
                    if (qr.off[i] >= 0) *reinterpret_cast<uint16_t *>(ep.aux_out + qr.off[i] + c0 + 8 * b + j2) = (uint16_t)w;
                }
        }
    }
    __syncwarp();
}

template <bool SLOPE, bool RESPF>
__device__ __forceinline__ void quad_tile_sgn(const LeanTile &lt, const QuadRows &qr, const LeanU &u, int64_t zp, int sgn,
                                              const EpiParams &ep, int32_t *out) {
    if (sgn == SGN_LO0) quad_tile<SLOPE, SGN_LO0, RESPF>(lt, qr, u, zp, ep, out);
    else if (sgn == SGN_HI0) quad_tile<SLOPE, SGN_HI0, RESPF>(lt, qr, u, zp, ep, out);
    else if (sgn == SGN_THR_HI) quad_tile<SLOPE, SGN_THR_HI, RESPF>(lt, qr, u, zp, ep, out);
    else quad_tile<SLOPE, SGN_THR_LO, RESPF>(lt, qr, u, zp, ep, out);
}

// ---- floating-point epilogue (kind::f16 path): v = acc + bias; act; [+ residual; post act]; cast -------------
// act codes: 0 none, 1 relu, 2 leaky-relu / PReLU with one slope.  out_type: 0 fp16, 1 bf16, 2 fp32.
struct FEpi {
    const float *bias;      // [N] or NULL
    const void *residual;   // [rows, N] in the OUTPUT dtype, or NULL
    float slope, post_slope;
    int act, post_act, out_type;
};
__device__ __forceinline__ float f_act(float v, int act, float slope) {
    return act == 1 ? fmaxf(v, 0.f) : (act == 2 ? (v < 0.f ? v * slope : v) : v);
}
__device__ __forceinline__ float f_load(const void *p, int64_t i, int t) {
    return t == 0 ? __half2float(((const __half *)p)[i]) : (t == 1 ? __bfloat162float(((const __nv_bfloat16 *)p)[i]) : ((const float *)p)[i]);
}
__device__ __forceinline__ void epi_chunk_f(const uint32_t (&acc)[EC], const int2 *chan, const FEpi &fe, const void *res,
                                            void *optr, int nvalid, bool vec) {
    float o[EC];
#pragma unroll
    for (int q = 0; q < EC; ++q) {
        float v = __uint_as_float(acc[q]) + __int_as_float(chan[q].x);
        v = f_act(v, fe.act, fe.slope);
        if (res) v += f_load(res, q < nvalid ? q : 0, fe.out_type);
        o[q] = f_act(v, fe.post_act, fe.post_slope);
    }
    if (vec && fe.out_type != 2) {  // nvalid is a multiple of 8 here
        uint32_t w[EC / 2];
#pragma unroll
        for (int t = 0; t < EC / 2; ++t) {
            if (fe.out_type == 0) { __half2 hv = __floats2half2_rn(o[2 * t], o[2 * t + 1]); w[t] = *reinterpret_cast<uint32_t *>(&hv); }
            else { __nv_bfloat162 bv = __floats2bfloat162_rn(o[2 * t], o[2 * t + 1]); w[t] = *reinterpret_cast<uint32_t *>(&bv); }
        }
        store_words<EC / 2>((char *)optr, w, nvalid * 2);
    } else if (vec) {
        uint32_t w[EC];
#pragma unroll
        for (int t = 0; t < EC; ++t) w[t] = __float_as_uint(o[t]);
        store_words<EC>((char *)optr, w, nvalid * 4);
    } else {
#pragma unroll
        for (int q = 0; q < EC; ++q) {
            if (q < nvalid) {
                if (fe.out_type == 0) ((__half *)optr)[q] = __float2half_rn(o[q]);
                else if (fe.out_type == 1) ((__nv_bfloat16 *)optr)[q] = __float2bfloat16_rn(o[q]);
                else ((float *)optr)[q] = o[q];
            }
        }
    }
}

// Warp roles of a CTA with EW epilogue warps (EW in {8, 12, 16}: 2, 3 or 4 column groups x 4 TMEM lane quarters):
// warps [0, EW) epilogue, [EW, EW+4) gather producers, EW+4 weight producer (TMA), EW+5 TMEM owner + MMA issuer.
// Fewer epilogue warps leave more issue slots (and registers: 128 / 96 / 80 per thread) to everyone else; the
// gather-heavy conv prefers 12, the epilogue-bound linears 16.
constexpr int EPI_WARPS_CONV = 12, EPI_WARPS_PAIRS = 16;
// Gather-producer warps: a thread per output row of the tile (the conv keeps each row's neighbour indices in registers).
constexpr int PROD_WARPS = TC_M / 32;

struct PMeta {  // per-tile metadata, double buffered
    uint32_t kmask;
    int32_t group, begin, end;
};

template <int STAGES>
struct PSmem {
    static size_t bytes(int n_tile, int rows_k) {
        return 1024 + (size_t)STAGES * (TC_M * TC_KB + (size_t)n_tile * TC_KB) + 2 * (size_t)rows_k * TC_M * 4 +
               (size_t)n_tile * 20 + 512;
    }
};

__device__ __forceinline__ void pairs_tile_lookup(const TcArgs &a, int tile_m, PMeta *m) {
    int g = 0, begin = tile_m * TC_M, end = a.n_pairs;
    if (a.offsets) {
        int t = tile_m;
        begin = end = -1;
        for (g = 0; g < a.n_groups; ++g) {
            int lo = a.offsets[g], hi = a.offsets[g + 1];
            int nt = (hi - lo + TC_M - 1) / TC_M;
            if (t < nt) { begin = lo + t * TC_M; end = hi; break; }
            t -= nt;
        }
    }
    // a tile past the last group (the grid covers an upper bound of the tile count) keeps begin = end = -1; its group index
    // must still be a valid one: the epilogue restages that group's (bias, mul) before it learns that the tile is empty
    // (reading one block past the end of the parameter arrays faulted when they ended a mapped region)
    m->group = g < a.n_groups ? g : a.n_groups - 1; m->begin = begin; m->end = end;
}

// KIND: 0 = int8 x int8 -> int32 (kind::i8, integer requant epilogue), 1 = fp16, 2 = bf16 (kind::f16, fp32
// accumulation, floating-point epilogue).  a.K is the contraction length in BYTES in every case.
// OUTK: which integer epilogue a kernel instance carries (chosen on the host from the epilogue descriptor).  One
// instance per output kind keeps the register allocation and the spills of each epilogue separate: with every path in
// one body the int8 linears lost 30 % to the pressure of the int32 quad code.
enum { OK_I8 = 0, OK_I16 = 1, OK_I32 = 2, OK_POST2 = 3 };

template <int MODE, int STAGES, int KIND, int EW, int OUTK>
__global__ void __launch_bounds__((EW + PROD_WARPS + 2) * 32, 1) igemm_tc_persistent(TcArgs a, const __grid_constant__ CUtensorMap tmap_w,
                                                                    EpiParams ep, FEpi fe, void *__restrict__ out, int tiles_m,
                                                                    int tiles_n) {
    constexpr int PW = PROD_WARPS, PT = PW * 32;  // producer warps / threads
    constexpr int P_EPI_WARPS = EW, P_PROD_WARP0 = EW, P_TMA_WARP = EW + PW, P_MMA_WARP = EW + PW + 1, P_THREADS = (EW + PW + 2) * 32;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int b_bytes = a.n_tile * TC_KB;
    constexpr int a_bytes = TC_M * TC_KB;
    uint8_t *sA = smem;
    uint8_t *sB = smem + STAGES * a_bytes;
    const int rows_k = MODE == 0 ? a.kvol : 2;
    int32_t *rows_s = (int32_t *)(sB + (size_t)STAGES * b_bytes);  // [2 slots][rows_k][128]
    int4 *chan4_s = (int4 *)(rows_s + 2 * rows_k * TC_M);         // [n_tile] (bias, mul, B, -B) of the current channel block
    int2 *chan_s = (int2 *)chan4_s;                               // float kinds: (bias bits, 0)
    int32_t *thr_s = (int32_t *)(chan4_s + a.n_tile);             // [n_tile] spare; words 0-1 hold the PReLU rounding addend (LeanU::k24)
    uint64_t *bars = (uint64_t *)(thr_s + a.n_tile);
    uint64_t *full = bars, *empty = bars + STAGES;
    uint64_t *meta_full = bars + 2 * STAGES, *tmem_full = meta_full + 2, *tmem_empty = tmem_full + 2;
    // xchg, peer_kmask and nt_flags are unused: the layout is kept because every change to it, even deleting the nt_flags
    // store below, alters register allocation and scheduling of all instances (DESIGN 3.5); compacting it needs a B200 A/B.
    uint64_t *xchg = tmem_empty + 2;  // [2] unused (only initialised)
    uint64_t *meta_empty = xchg + 2;  // every reader of meta[slot] / rows[slot] of the slot's previous tile has taken its copy
    PMeta *meta = (PMeta *)(meta_empty + 2);
    uint32_t *tmem_ptr = (uint32_t *)(meta + 2);
    uint32_t *lean_off = tmem_ptr + 1;  // set once a staged channel block fails the lean-epilogue preconditions
    uint32_t *peer_kmask = lean_off + 1;  // [2] unused
    uint32_t *nt_flags = peer_kmask + 2;  // [16] unused (zeroed only)
    const int tile0 = (int)blockIdx.x, tile_step = (int)gridDim.x;  // tiles of this CTA: tile0, tile0 + tile_step, ...

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_chunks = (a.K + TC_KB - 1) / TC_KB;
    const int total_tiles = tiles_m * tiles_n;

    if (warp == P_MMA_WARP && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], PT + 1);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&meta_full[b], PT);
            mbar_init(&tmem_full[b], 1);
            mbar_init(&tmem_empty[b], P_EPI_WARPS);
            mbar_init(&xchg[b], 1);
            mbar_init(&meta_empty[b], P_EPI_WARPS + 2);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == P_TMA_WARP && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w) : "memory");
    if (warp == P_MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"((uint32_t)(2 * a.tmem_cols)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // per-channel epilogue constants of a single channel block are staged once (grouped weights reload per tile)
    const bool chan_static = tiles_n == 1 && !(MODE == 1 && a.bias_per_group);
    const int64_t zp_all = KIND == 0 ? ep.zp[0] : 0;
    int64_t vmax = 0;
    const int sgn_mode = KIND == 0 ? lean_mode(ep, zp_all, (int64_t)a.K * (MODE == 0 ? a.kvol : 1), ep.row_bias_bound, &vmax) : SGN_NONE;
    if (tid >= 32 && tid < 48) nt_flags[tid - 32] = 0u;  // unused (see the carve-up above)
    if (tid == 0) {
        *lean_off = sgn_mode != SGN_NONE ? 0u : 1u;
        thr_s[0] = (1 << 24) - 1; thr_s[1] = 0;
        if (KIND == 0 && ep.post_mul) {  // second-stage constants of the lean path (LeanU::post2_addr)
            const Post2 p2 = load_post2(ep);
            int64_t t2 = 0;
            if (p2.mul) { const int64_t nz = -p2.zp, m = (int64_t)p2.mul; t2 = nz >= 0 ? (nz + m - 1) / m : -((-nz) / m); }
            const int64_t c02 = p2.zp + (p2.shift > 0 ? (int64_t)1 << (p2.shift - 1) : 0);
            thr_s[4] = (int32_t)p2.mul;
            thr_s[5] = (int32_t)(t2 > 2147483647ll ? 2147483647ll : (t2 < -2147483648ll ? -2147483648ll : t2));
            thr_s[6] = p2.slope; thr_s[7] = p2.shift >= 32 ? p2.shift - 32 : 0;
            thr_s[8] = (int32_t)(uint32_t)c02; thr_s[9] = (int32_t)(uint32_t)((uint64_t)c02 >> 32);
            thr_s[10] = (p2.shift >= 32 && !tie_possible(p2.mul, p2.zp, p2.shift, (int64_t)1 << 31)) ? 1 : 0;
        }
    }
    __syncthreads();
    if (chan_static)
        for (int cb = warp * 32; cb < a.n_tile; cb += P_THREADS) {  // per-warp form kept: `c = tid; c += P_THREADS` changes the SASS
            const int c = cb + lane;
            const bool valid = c < a.n_tile;
            if (KIND == 0) {
                const int32_t b = c < a.N && ep.bias ? ep.bias[c] : 0;
                const uint32_t mu = c < a.N ? ep.mul[ep.mul_is_scalar ? 0 : c] : 0u;
                if (valid) {
                    const bool ok = stage_channel(b, mu, zp_all, ep.shift, ep.out_type, vmax, &chan4_s[c]);
                    if (!ok && sgn_mode != SGN_NONE) atomicOr(lean_off, 1u);
                }
            } else if (valid) {
                chan_s[c] = make_int2(c < a.N && fe.bias ? __float_as_int(fe.bias[c]) : 0, 0);
            }
        }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp >= P_PROD_WARP0 && warp < P_PROD_WARP0 + PW) {
        // ================= metadata + gather producers =================
        const int r = tid - P_PROD_WARP0 * 32;
        int it = 0;       // running pipeline step across tiles
        int j = 0;        // local tile counter
        // The neighbour rows of a tile are fetched one tile ahead into registers: the 27 dependent-latency loads
        // overlap the previous tile's gathers instead of stalling the pipeline at every tile boundary.
        constexpr int PRE = 27;
        int32_t nv[PRE];
        const bool pre = MODE == 0 && a.kvol <= PRE;
        auto fetch = [&](int t) {
            const int m = (t / tiles_n) * TC_M + r;
            const bool ok = t < total_tiles && m < a.n_out;
#pragma unroll
            for (int u = 0; u < PRE; ++u) nv[u] = (ok && u < a.kvol) ? __ldg(&a.nbr[(int64_t)u * a.ld + m]) : 0;
        };
        if (pre) fetch(tile0);
        for (int tile = tile0; tile < total_tiles; tile += tile_step, ++j) {
            const int slot = j & 1;
            const int tile_m = tile / tiles_n;
            int32_t *rows = rows_s + slot * rows_k * TC_M;
            if (r == 0) TRACE(j, 0);
            // The metadata slot is free once every reader of tile j-2 has taken its copy (the epilogue warps do that when
            // they START tile j-2): the gathers of tile j run while the epilogue of tile j-2 still drains its accumulator;
            // only the MMA issuer waits for tmem_empty.  (Waiting for tmem_empty here put meta + gather latency of every
            // tile on the critical path: period = (fill + MMA + epilogue) / 2, measured with FPCC_TC_TRACE.)
            mbar_wait(&meta_empty[slot], ((j >> 1) & 1) ^ 1);
            if (r == 0) TRACE(j, 1);
            if (r == 0) meta[slot].kmask = 0;
            asm volatile("bar.sync 1, %0;" ::"n"(PT) : "memory");
            if (MODE == 0) {
                const int m = tile_m * TC_M + r;
                uint32_t mine = 0;
                if (pre) {
#pragma unroll
                    for (int u = 0; u < PRE; ++u)
                        if (u < a.kvol) {
                            rows[u * TC_M + r] = nv[u] - 1;
                            mine |= (uint32_t)(nv[u] != 0) << u;
                        }
                    fetch(tile + tile_step);
                } else {
                    for (int k = 0; k < a.kvol; ++k) {
                        int32_t v = m < a.n_out ? __ldg(&a.nbr[(int64_t)k * a.ld + m]) : 0;
                        rows[k * TC_M + r] = v - 1;
                        mine |= (uint32_t)(v != 0) << k;
                    }
                }
                mine = __reduce_or_sync(0xffffffffu, mine);
                if (lane == 0 && mine) atomicOr(&meta[slot].kmask, mine);
            } else {
                if (r == 0) { pairs_tile_lookup(a, tile_m, &meta[slot]); }
                asm volatile("bar.sync 1, %0;" ::"n"(PT) : "memory");
                const int p = meta[slot].begin + r;
                const bool ok = meta[slot].begin >= 0 && p < meta[slot].end;
                rows[r] = ok ? (a.in_idx ? __ldg(&a.in_idx[p]) : p) : -1;
                rows[TC_M + r] = ok ? (a.out_idx ? __ldg(&a.out_idx[p]) : p) : -1;
                if (r == 0) meta[slot].kmask = meta[slot].begin >= 0 && meta[slot].begin < meta[slot].end ? 1u : 0u;
            }
            __threadfence_block();
            mbar_arrive(&meta_full[slot]);
            mbar_wait(&meta_full[slot], (j >> 1) & 1);
            uint32_t rem = meta[slot].kmask;
            const int total = __popc(rem) * n_chunks;
            int k = 0, kc = n_chunks - 1;
            if (r == 0) TRACE(j, 2);
            for (int i = 0; i < total; ++i, ++it) {
                if (++kc == n_chunks) { kc = 0; k = __ffs(rem) - 1; rem &= rem - 1; }
                const int stage = it % STAGES;
                mbar_wait(&empty[stage], ((it / STAGES) & 1) ^ 1);
                // 8 consecutive lanes fetch the 8 16-byte pieces of ONE row (a full 128-byte line), 4 rows per
                // instruction: 4 L1 wavefronts per LDGSTS instead of 32 with one row per lane.
                // This lane serves rows base..base+7 (two 16-byte shared loads fetch their source rows).
                const int base = (r & ~31) + (lane >> 3) * 8;
                const uint32_t rk = smem_u32(rows + (MODE == 0 ? k : 0) * TC_M + base);
                const int4 s0 = lds128(rk), s1 = lds128(rk + 16);
                const int32_t srcs[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
                const int piece = lane & 7;
                const bool k_ok = kc * TC_KB + piece * 16 < a.K;
                const uint32_t dst0 = smem_u32(sA + stage * a_bytes);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int32_t src = srcs[i];
                    const int row = base + i;
                    const bool ok = src >= 0 && k_ok;
                    const int8_t *gsrc = a.A + (ok ? (int64_t)src * a.K + kc * TC_KB + piece * 16 : 0);
                    cp_async16(dst0 + row * TC_KB + ((piece ^ (row & 7)) << 4), gsrc, ok ? 16u : 0u);
                }
                // The stage's full barrier is signalled by the copy engine itself once this thread's copies have
                // landed (no commit/wait lag in the producer): all STAGES stages can be in flight or queued.
                asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&full[stage])) : "memory");
            }
        }
    } else if (warp == P_TMA_WARP) {
        // ================= weight producer (TMA) =================
        if (lane == 0) {
            int it = 0, j = 0;
            for (int tile = tile0; tile < total_tiles; tile += tile_step, ++j) {
                const int slot = j & 1;
                const int n0 = (tile % tiles_n) * a.n_tile;
                mbar_wait(&meta_full[slot], (j >> 1) & 1);
                uint32_t rem = meta[slot].kmask;
                const int total = __popc(rem) * n_chunks;
                const int group = MODE == 1 ? meta[slot].group : 0;
                mbar_arrive(&meta_empty[slot]);
                int k = 0, kc = n_chunks - 1;
                for (int i = 0; i < total; ++i, ++it) {
                    if (++kc == n_chunks) { kc = 0; k = __ffs(rem) - 1; rem &= rem - 1; }
                    const int stage = it % STAGES;
                    mbar_wait(&empty[stage], ((it / STAGES) & 1) ^ 1);
                    mbar_expect_tx(&full[stage], (uint32_t)b_bytes);
                    const int wrow = (MODE == 0 ? k : group) * a.N + n0;
                    tma_load_2d(smem_u32(sB + (size_t)stage * b_bytes), &tmap_w, &full[stage], kc * TC_KB, wrow);
                }
            }
        }
    } else if (warp == P_MMA_WARP) {
        // ================= MMA issuer =================
        if (lane == 0) {
            const uint32_t idesc = KIND == 0 ? umma_idesc_i8(a.n_tile) : umma_idesc_f16(a.n_tile, KIND == 2);
            int it = 0, j = 0;
            for (int tile = tile0; tile < total_tiles; tile += tile_step, ++j) {
                const int slot = j & 1;
                mbar_wait(&meta_full[slot], (j >> 1) & 1);
                const int total = __popc(meta[slot].kmask) * n_chunks;
                mbar_arrive(&meta_empty[slot]);
                mbar_wait(&tmem_empty[slot], ((j >> 1) & 1) ^ 1);  // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t tacc = tmem_base + (uint32_t)(slot * a.tmem_cols);
                for (int i = 0; i < total; ++i, ++it) {
                    const int stage = it % STAGES;
                    mbar_wait(&full[stage], (it / STAGES) & 1);
                    if (i == 0) TRACE(j, 3);
                    fence_proxy_async();  // the gathered rows were written through the generic proxy (cp.async)
                    tc_fence_after();
                    const uint64_t ad = umma_desc_sw128(smem_u32(sA + stage * a_bytes));
                    const uint64_t bd = umma_desc_sw128(smem_u32(sB + (size_t)stage * b_bytes));
#pragma unroll
                    for (int q = 0; q < TC_KB / 32; ++q) {  // 32 bytes of K per instruction for both kinds
                        if (KIND == 0) umma_i8(tacc, ad + 2 * q, bd + 2 * q, idesc, (uint32_t)(i > 0 || q > 0));
                        else umma_f16(tacc, ad + 2 * q, bd + 2 * q, idesc, (uint32_t)(i > 0 || q > 0));
                    }
                    umma_commit(&empty[stage]);
                }
                TRACE(j, 4);
                if (total > 0) umma_commit(&tmem_full[slot]);
                else mbar_arrive(&tmem_full[slot]);
            }
        }
    } else if (warp < P_EPI_WARPS) {
        // ================= epilogue =================
        const int quarter = warp & 3, group = warp >> 2;  // TMEM lane quarter, column group (4 groups of 4 warps)
        const int r = quarter * 32 + lane;  // tile row == TMEM lane
        const bool has_slope = KIND == 0 && ep.slope != nullptr, has_post = KIND == 0 && ep.post_slope != nullptr;
        const int32_t slope = has_slope ? ep.slope[0] : 0, post = has_post ? ep.post_slope[0] : 0;
        const int64_t zp = KIND == 0 ? ep.zp[0] : 0;
        const int shift = ep.shift;
        const int cols_grp = (((a.n_tile + P_EPI_WARPS / 4 - 1) / (P_EPI_WARPS / 4) + EC - 1) / EC) * EC;  // columns per group, multiple of EC
        const int c_begin = min(a.n_tile, group * cols_grp), c_end = min(a.n_tile, c_begin + cols_grp);
        const bool out_al = ((uintptr_t)out & 15) == 0 && (ep.out_ld & 15) == 0;
        LeanU lu;
        {
            const int64_t c0v = zp + (shift > 0 ? (int64_t)1 << (shift - 1) : 0);
            lu.slope = slope; lu.post = post; lu.shift = shift; { const uint32_t ka = smem_u32(thr_s); int32_t k_lo, k_hi; asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(k_lo), "=r"(k_hi) : "r"(ka)); lu.k24 = pack64((uint32_t)k_lo, (uint32_t)k_hi); }
            lu.c0_lo = (uint32_t)c0v; lu.c0_hi = (uint32_t)((uint64_t)c0v >> 32);
            lu.ovf_add = shift > 0 && shift <= 31 ? 1u << (shift - 1) : 0u;
            lu.ovf_lim = shift <= 31 ? (1u << shift) - 1u : 0xffffffffu;
        }
        lu.post2_addr = smem_u32(thr_s + 4);
        const bool post2_on = KIND == 0 && OUTK == OK_POST2;
        // Output rows of grouped convs (row_perm): fetched ONE TILE AHEAD -- the dependent global load sat on the tile
        // boundary of every epilogue warp (~1 us per tile in the FPCC_TC_TRACE timeline).
        const bool use_perm = MODE == 0 && a.row_perm != nullptr;
        constexpr bool QUAD = KIND == 0 && OUTK == OK_I32;
        int32_t pm_next = 0, qpm_next[4] = {0, 0, 0, 0};
        auto perm_fetch = [&](int t) {
            if (t >= total_tiles) return;
            const int64_t base = (int64_t)(t / tiles_n) * TC_M;
            if (base + r < a.n_out) pm_next = __ldg(&a.row_perm[base + r]);
            if (QUAD) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int64_t mti = base + quarter * 32 + (lane >> 2) + 8 * i;
                    if (mti < a.n_out) qpm_next[i] = __ldg(&a.row_perm[mti]);
                }
            }
        };
        if (use_perm) perm_fetch(tile0);
        int j = 0;
        for (int tile = tile0; tile < total_tiles; tile += tile_step, ++j) {
            const int slot = j & 1;
            const int tile_m = tile / tiles_n, n0 = (tile % tiles_n) * a.n_tile;
            const int32_t pm = pm_next;
            int32_t qpm[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) qpm[i] = qpm_next[i];
            if (use_perm) perm_fetch(tile + tile_step);
            mbar_wait(&meta_full[slot], (j >> 1) & 1);
            const bool have_acc = meta[slot].kmask != 0;
            const int pbase = (MODE == 1 && a.bias_per_group) ? meta[slot].group * a.N : 0;
            // grouped weights / several channel blocks: restage (bias, mul) of this tile's block, on every tile.  Restaging
            // only when the block changes measured SLOWER on B200 -- selection linear with the fused second stage 0.203 ->
            // 0.310 ms: without the two CTA-wide barriers per tile the 16 epilogue warps reach the accumulator wait early and
            // their mbarrier polls take issue slots from the four gather-producer warps these kernels are bound by
            // (profiles/r02_sel_linear_variants.txt).
            if (!chan_static) {
                asm volatile("bar.sync 2, %0;" ::"n"(P_EPI_WARPS * 32) : "memory");  // every epilogue warp is done with the previous tile's values
                const int t = warp * 32 + lane;
                if (warp * 32 < a.n_tile) {  // n_tile <= 256 <= 32 * epilogue warps
                    const bool valid = t < a.n_tile;
                    const int pc = pbase + min(n0 + t, a.N - 1);
                    if (KIND == 0) {
                        const int32_t b = ep.bias ? __ldg(&ep.bias[pc]) : 0;
                        const uint32_t mu = __ldg(&ep.mul[ep.mul_is_scalar ? 0 : pc]);
                        if (valid) {
                            const bool ok = stage_channel(b, mu, zp_all, ep.shift, ep.out_type, vmax, &chan4_s[t]);
                            if (!ok && sgn_mode != SGN_NONE) atomicOr(lean_off, 1u);
                        }
                    } else if (valid) {
                        chan_s[t] = make_int2(fe.bias ? __float_as_int(__ldg(&fe.bias[pc])) : 0, 0);
                    }
                }
                asm volatile("bar.sync 2, %0;" ::"n"(P_EPI_WARPS * 32) : "memory");
            }
            const int32_t *rows = rows_s + slot * rows_k * TC_M;
            const int64_t mt = (int64_t)tile_m * TC_M + r;  // MODE 0: column of the neighbour table
            const bool row_ok = MODE == 0 ? (mt < a.n_out) : (rows[TC_M + r] >= 0);
            const int64_t m = MODE == 0 ? ((use_perm && row_ok) ? (int64_t)pm : mt) : (int64_t)rows[TC_M + r];
            if (KIND == 0 && ep.residual && row_ok) {
                // residual rows of this tile: start them towards L2 while the MMAs of the tile are still running
                const char *rp = (const char *)(ep.residual + m * a.N + n0 + c_begin);
                for (int off = 0; off < (c_end - c_begin) * 4; off += 128)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + off));
            }
            // int32 rows: quad layout (whole sectors per access); rows q, q+8, q+16, q+24 of the warp's quarter
            QuadRows qr;
            if (KIND == 0 && OUTK == OK_I32) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int rr = quarter * 32 + (lane >> 2) + 8 * i;
                    int64_t mm;
                    bool ok;
                    if (MODE == 0) {
                        const int64_t mti = (int64_t)tile_m * TC_M + rr;
                        ok = mti < a.n_out;
                        mm = (use_perm && ok) ? (int64_t)qpm[i] : mti;
                    } else {
                        mm = (int64_t)rows[TC_M + rr];
                        ok = mm >= 0;
                    }
                    qr.off[i] = ok ? mm * a.N + n0 : -1;
                    qr.rb[i] = (ep.row_bias && ok) ? (int32_t)__ldg(&ep.row_idx[mm]) : 0;
                }
            }
            // this warp holds its copies of meta[slot] / rows[slot]: the producers may build tile j+2 in the slot
            __syncwarp();
            if (lane == 0) mbar_arrive(&meta_empty[slot]);
            mbar_wait(&tmem_full[slot], (j >> 1) & 1);
            tc_fence_after();
            if (tid == 0) TRACE(j, 5);
            const uint32_t tacc = tmem_base + (uint32_t)(slot * a.tmem_cols) + ((uint32_t)(quarter * 32) << 16);
            const bool lean = KIND == 0 && OUTK != OK_I16 && out_al && (a.N & 15) == 0 && *(volatile uint32_t *)lean_off == 0u && !(post2_on && has_slope);
            if (KIND == 0 && lean) {
                LeanTile lt;
                lt.tacc = tacc; lt.chan_addr = smem_u32(chan4_s); lt.c_begin = c_begin; lt.c_end = c_end; lt.ncols = a.N - n0; lt.n0 = n0; lt.ncols_total = a.N;
                lt.have_acc = have_acc; lt.row_ok = row_ok; lt.has_post = has_post; lt.al32 = MODE == 0 && ((uintptr_t)out & 31) == 0 && (ep.out_ld & 31) == 0;
                const int64_t row0 = row_ok ? m * a.N + n0 : 0;
                // int8 rows may go to a column slice of a wider buffer (fpcc_epilogue::out_ld: row pitch in elements)
                const int64_t ld8 = ep.out_ld > 0 ? ep.out_ld : a.N;
                lt.orow = (ep.out_type == FPCC_OUT_I8 || post2_on) ? (char *)out + (row_ok ? m * ld8 + n0 : 0) : (char *)out + row0 * 4;
                lt.rb_row = ep.row_bias ? ep.row_bias + (row_ok ? (int64_t)__ldg(&ep.row_idx[m]) * a.N + n0 : 0) : nullptr;
                lt.res_row = ep.residual ? ep.residual + row0 : nullptr;
                lt.aux_row = (OUTK == OK_I32 && ep.aux_out) ? ep.aux_out + row0 : nullptr;
                if (OUTK == OK_I8) {
                    if (has_slope) lean_tile_sgn<FPCC_OUT_I8, true, false, false, false>(lt, lu, zp, sgn_mode, ep);
                    else lean_tile_sgn<FPCC_OUT_I8, false, false, false, false>(lt, lu, zp, sgn_mode, ep);
                } else if (OUTK == OK_I32) {
                    if (has_slope) quad_tile_sgn<true, false>(lt, qr, lu, zp, sgn_mode, ep, (int32_t *)out);
                    else quad_tile_sgn<false, MODE == 0>(lt, qr, lu, zp, sgn_mode, ep, (int32_t *)out);
                } else if (OUTK == OK_POST2) {
                    // selection linears of the multi-step predictors / conv2 of a ResBlock: no PReLU of their own
                    if (ep.post_slope2 != nullptr) lean_tile_sgn<FPCC_OUT_I32, false, true, true, false>(lt, lu, zp, sgn_mode, ep);
                    else lean_tile_sgn<FPCC_OUT_I32, false, true, false, false>(lt, lu, zp, sgn_mode, ep);
                }
            } else
            for (int c0 = c_begin; c0 < c_end; c0 += EC) {
                uint32_t acc[EC];
                __syncwarp();
                if (have_acc) {
                    tmem_ld16(tacc + (uint32_t)c0, acc);
                } else {
#pragma unroll
                    for (int q = 0; q < EC; ++q) acc[q] = 0;
                }
                const int nb = n0 + c0;
                if (!row_ok || nb >= a.N) continue;
                if (KIND != 0) {
                    const int esz = fe.out_type == 2 ? 4 : 2;
                    const int nvalid = min(EC, a.N - nb);
                    const void *res = fe.residual ? (const char *)fe.residual + (m * a.N + nb) * esz : nullptr;
                    epi_chunk_f(acc, chan_s + c0, fe, res, (char *)out + (m * a.N + nb) * esz, nvalid,
                                out_al && (a.N & 7) == 0);
                    continue;
                }
                EpiCtx cx;
                cx.chan4 = chan4_s + c0;
                cx.slope = slope; cx.post = post; cx.zp = zp; cx.shift = shift;
                cx.half = shift > 0 ? (int64_t)1 << (shift - 1) : 0; cx.sgn = shift > 0;
                cx.row_bias = ep.row_bias ? ep.row_bias + (int64_t)__ldg(&ep.row_idx[m]) * a.N + nb : nullptr;
                cx.residual = ep.residual ? ep.residual + m * a.N + nb : nullptr;
                cx.has_post = has_post;
                cx.nvalid = min(EC, a.N - nb);
                void *optr = (ep.out_type == FPCC_OUT_I8 || post2_on) ? (void *)((char *)out + m * (ep.out_ld > 0 ? (int64_t)ep.out_ld : (int64_t)a.N) + nb)
                                                                      : (void *)((char *)out + (m * a.N + nb) * (ep.out_type == FPCC_OUT_I16 ? 2 : 4));
                const bool vec = out_al && (a.N & 15) == 0;
                const bool rb = ep.row_bias != nullptr;
                Post2 p2;
                p2.on = false; p2.dual = false;
                if (post2_on || (OUTK == OK_I32 && ep.aux_out)) p2 = load_post2(ep);
                cx.aux = p2.dual ? ep.aux_out + m * a.N + nb : nullptr;
                if (OUTK == OK_I8) epi_dispatch<FPCC_OUT_I8>(acc, cx, optr, vec, has_slope, rb, p2);
                else if (OUTK == OK_I32 || OUTK == OK_POST2) epi_dispatch<FPCC_OUT_I32>(acc, cx, optr, vec, has_slope, rb, p2);
                else epi_dispatch<FPCC_OUT_I16>(acc, cx, optr, vec, has_slope, rb, p2);
            }
            tc_fence_before();
            __syncwarp();
            if (tid == 0) TRACE(j, 6);
            if (lane == 0) mbar_arrive(&tmem_empty[slot]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == P_MMA_WARP) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * a.tmem_cols)) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------
// tensor-pipe ceiling probe: back-to-back kind::i8 MMAs (M=128, N=256, K=32) on resident smem tiles, no
// loads in the loop.  Gives the measured int8 peak that the roofline of this kernel is quoted against.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128, 1) mma_i8_peak_kernel(int iters, int n) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t done;
    __shared__ uint32_t tmem_ptr;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < (TC_M * TC_KB + 256 * TC_KB) / 4; i += blockDim.x) ((uint32_t *)smem)[i] = 0x01010101u;
    if (threadIdx.x == 0) {
        mbar_init(&done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_ptr)), "r"(256u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_ptr;
    if (warp == 1 && lane == 0) {
        const uint32_t idesc = umma_idesc_i8(n);
        const uint64_t ad = umma_desc_sw128(smem_u32(smem));
        const uint64_t bd = umma_desc_sw128(smem_u32(smem + TC_M * TC_KB));
        for (int i = 0; i < iters; ++i) {
#pragma unroll
            for (int j = 0; j < 4; ++j) umma_i8(tmem_base, ad + 2 * j, bd + 2 * j, idesc, 1u);
        }
        umma_commit(&done);
    }
    mbar_wait(&done, 0);
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u) : "memory");
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int g_tc_mode = -1;  // -1: read FPCC_TC from the environment on first use
static int g_sm_budget = 0;  // persistent GEMM grids use at most this many SMs (0 = all)

bool tc_enabled() {
    if (g_tc_mode < 0) {
        const char *e = getenv("FPCC_TC");
        g_tc_mode = (e && e[0] == '0') ? 0 : 1;
    }
    return g_tc_mode == 1;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// weights are static per layer: one descriptor per (pointer, rows, K, box rows)
static int weight_tensor_map(const int8_t *w, int64_t rows, int K, int box_rows, CUtensorMap *out) {
    static std::mutex mu;
    static std::map<std::tuple<const void *, int64_t, int, int>, CUtensorMap> cache;
    std::lock_guard<std::mutex> lk(mu);
    auto key = std::make_tuple((const void *)w, rows, K, box_rows);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return FPCC_OK; }
    EncodeTiledFn fn = encode_fn();
    FPCC_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)K};
    cuuint32_t box[2] = {(cuuint32_t)TC_KB, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUtensorMap m;
    CUresult r = fn(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void *)w, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FPCC_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d (rows %lld, K %d, box %d)", (int)r, (long long)rows, K, box_rows);
    if (cache.size() > 4096) cache.clear();
    cache[key] = m;
    *out = m;
    return FPCC_OK;
}

static bool tc_shape_ok(const void *A, const void *W, int K, int N) {
    return K >= 32 && K % 16 == 0 && N >= 16 && (((uintptr_t)A | (uintptr_t)W) & 15) == 0;
}

static int pick_tile(int N, int *n_tile, int *tmem_cols) {
    int nt = N >= 256 ? 256 : ((N + 15) / 16) * 16;
    int cols = 32;
    while (cols < nt) cols <<= 1;
    *n_tile = nt;
    *tmem_cols = cols;
    return (N + nt - 1) / nt;
}

constexpr size_t TC_SMEM_MAX = 227 * 1024;
template <int MODE, int STAGES, int KIND, int OUTK>
static int launch_outk(const TcArgs &a, const CUtensorMap &tmap, const EpiParams &ep, const FEpi &fe, void *out, int tiles_m,
                       int n_blocks_n, int grid, size_t smem, cudaStream_t s) {
    // Epilogue warps per kernel instance.  The register file splits over four sub-partitions: 12 + 6 warps get 96 registers
    // per thread, 16 + 6 warps 80, 8 + 6 warps 128.  The int32-output instances (quad layout, residual prefetch) spill at 96 / 80
    // and run faster on FEWER warps with more registers (ResBlock conv2: 0.354 -> 0.307 ms with 8, 0.371 ms with 16;
    // profiles/r02_epilogue_warps.txt).
    constexpr bool I32_OUT = KIND == 0 && (OUTK == OK_I32 || OUTK == OK_POST2);
    constexpr int EW = I32_OUT ? 8 : (MODE == 0 ? EPI_WARPS_CONV : EPI_WARPS_PAIRS);
    constexpr int OK = KIND == 0 ? OUTK : OK_I8;
    constexpr int THREADS = (EW + PROD_WARPS + 2) * 32;
    auto kern = igemm_tc_persistent<MODE, STAGES, KIND, EW, OK>;
    static bool configured = false;
    if (!configured) {
        FPCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_MAX));
        configured = true;
    }
    kern<<<grid, THREADS, smem, s>>>(a, tmap, ep, fe, out, tiles_m, n_blocks_n);
    FPCC_LAUNCH_CHECK();
    return FPCC_OK;
}

template <int MODE, int STAGES, int KIND>
static int launch_stages(const TcArgs &a, const CUtensorMap &tmap, const EpiParams &ep, const FEpi &fe, void *out, int tiles_m,
                         int n_blocks_n, int grid, int rows_k, cudaStream_t s) {
    size_t smem = PSmem<STAGES>::bytes(a.n_tile, rows_k);
    FPCC_REQUIRE(smem <= TC_SMEM_MAX, "igemm_tc: %zu bytes of shared memory exceed the 227 KB limit", smem);
    if (KIND != 0) return launch_outk<MODE, STAGES, KIND, OK_I8>(a, tmap, ep, fe, out, tiles_m, n_blocks_n, grid, smem, s);
    if (ep.post_mul && !ep.aux_out) return launch_outk<MODE, STAGES, KIND, OK_POST2>(a, tmap, ep, fe, out, tiles_m, n_blocks_n, grid, smem, s);
    if (ep.out_type == FPCC_OUT_I8) return launch_outk<MODE, STAGES, KIND, OK_I8>(a, tmap, ep, fe, out, tiles_m, n_blocks_n, grid, smem, s);
    if (ep.out_type == FPCC_OUT_I32) return launch_outk<MODE, STAGES, KIND, OK_I32>(a, tmap, ep, fe, out, tiles_m, n_blocks_n, grid, smem, s);
    return launch_outk<MODE, STAGES, KIND, OK_I16>(a, tmap, ep, fe, out, tiles_m, n_blocks_n, grid, smem, s);
}

template <int MODE, int KIND>
static int launch_tc(TcArgs &a, const void *W, int64_t w_rows, int tiles_m, const EpiParams &ep, const FEpi &fe, void *out,
                     cudaStream_t s) {
    int n_blocks_n = pick_tile(a.N, &a.n_tile, &a.tmem_cols);
    const int rows_k = MODE == 0 ? a.kvol : 2;
    int total = tiles_m * n_blocks_n;
    int sms = g_sm_budget > 0 && g_sm_budget < sm_count() ? g_sm_budget : sm_count();
    CUtensorMap tmap;
    int rc = weight_tensor_map((const int8_t *)W, w_rows, a.K, a.n_tile, &tmap);
    if (rc) return rc;
    int grid = total < sms ? total : sms;
    // four operand stages where they fit in shared memory, three otherwise (wide tiles with many kernel offsets)
    if (PSmem<4>::bytes(a.n_tile, rows_k) <= TC_SMEM_MAX)
        return launch_stages<MODE, 4, KIND>(a, tmap, ep, fe, out, tiles_m, n_blocks_n, grid, rows_k, s);
    return launch_stages<MODE, 3, KIND>(a, tmap, ep, fe, out, tiles_m, n_blocks_n, grid, rows_k, s);
}

int launch_conv_tc(const int8_t *feats, int n_in, int c_in, const int8_t *weight, int kvol, int c_out, const int32_t *nbr,
                   int64_t ld, int n_out, const int32_t *row_perm, const EpiParams &ep, void *out, cudaStream_t s) {
    (void)n_in;
    if (!tc_shape_ok(feats, weight, c_in, c_out) || kvol > TC_MAX_KVOL) return FPCC_ERR_UNSUPPORTED;
    TcArgs a = {};
    a.A = feats; a.K = c_in; a.N = c_out;
    a.nbr = nbr; a.ld = ld; a.n_out = n_out; a.kvol = kvol; a.row_perm = row_perm;
    FEpi fe = {};
    return launch_tc<0, 0>(a, weight, (int64_t)kvol * c_out, ceil_div(n_out, TC_M), ep, fe, out, s);
}

int launch_pairs_tc(const PairArgs &p, const EpiParams &ep, void *out, int max_tiles, cudaStream_t s) {
    (void)max_tiles;
    if (p.raw != 0 || !tc_shape_ok(p.A, p.W, p.K, p.N)) return FPCC_ERR_UNSUPPORTED;
    TcArgs a = {};
    a.A = p.A; a.K = p.K; a.N = p.N;
    a.in_idx = p.in_idx; a.out_idx = p.out_idx; a.offsets = p.offsets;
    a.n_groups = p.n_groups; a.n_pairs = p.n_pairs; a.bias_per_group = p.bias_per_group;
    int tiles = ceil_div(p.n_pairs, TC_M) + (p.offsets ? p.n_groups : 0);
    FEpi fe = {};
    return launch_tc<1, 0>(a, p.W, (int64_t)p.n_groups * p.N, tiles, ep, fe, out, s);
}

}  // namespace fpcc

// ---- fp16 / bf16 entry points (MinkowskiEngine / torchsparse float layers) ---------------------------------
static int f16_common(int dtype, int out_type, int act, int post_act, int c_in, int c_out, const void *A, const void *W, const void *out) {
    FPCC_REQUIRE(dtype == 0 || dtype == 1, "f16 GEMM: dtype must be 0 (fp16) or 1 (bf16)");
    FPCC_REQUIRE(out_type >= 0 && out_type <= 2, "f16 GEMM: out_type must be 0 (fp16), 1 (bf16) or 2 (fp32)");
    FPCC_REQUIRE(act >= 0 && act <= 2 && post_act >= 0 && post_act <= 2, "f16 GEMM: bad activation code");
    FPCC_REQUIRE(c_in >= 16 && c_in % 8 == 0 && c_out >= 16, "f16 GEMM: needs C_in %% 8 == 0, C_in >= 16, C_out >= 16 (got %d -> %d)", c_in, c_out);
    FPCC_REQUIRE((((uintptr_t)A | (uintptr_t)W | (uintptr_t)out) & 15) == 0, "f16 GEMM: pointers must be 16-byte aligned");
    return FPCC_OK;
}

extern "C" int fpcc_spconv_f16(const void *feats, int dtype, int n_in, int c_in, const void *weight, int kvol, int c_out,
                               const int32_t *nbr_table, int64_t ld, int n_out, const int32_t *row_perm, const float *bias, int act, float slope,
                               const void *residual, int post_act, float post_slope, void *out, int out_type, void *stream) {
    using namespace fpcc;
    FPCC_REQUIRE(feats && weight && nbr_table && out, "spconv_f16: NULL pointer");
    FPCC_REQUIRE(n_in > 0 && n_out > 0 && kvol > 0 && kvol <= TC_MAX_KVOL && ld >= n_out, "spconv_f16: bad sizes");
    int rc = f16_common(dtype, out_type, act, post_act, c_in, c_out, feats, weight, out);
    if (rc) return rc;
    TcArgs a = {};
    a.A = (const int8_t *)feats; a.K = 2 * c_in; a.N = c_out;
    a.nbr = nbr_table; a.ld = ld; a.n_out = n_out; a.kvol = kvol; a.row_perm = row_perm;
    FEpi fe = {bias, residual, slope, post_slope, act, post_act, out_type};
    EpiParams ep = {};
    if (dtype == 0) return launch_tc<0, 1>(a, weight, (int64_t)kvol * c_out, ceil_div(n_out, TC_M), ep, fe, out, (cudaStream_t)stream);
    return launch_tc<0, 2>(a, weight, (int64_t)kvol * c_out, ceil_div(n_out, TC_M), ep, fe, out, (cudaStream_t)stream);
}

extern "C" int fpcc_linear_f16(const void *A, int dtype, int m, int k, const void *W, int n, const int32_t *sel_row,
                               const int32_t *sel_out, const int32_t *sel_offsets, int n_groups, int n_sel, const float *bias,
                               int act, float slope, const void *residual, int post_act, float post_slope, void *out,
                               int out_type, void *stream) {
    using namespace fpcc;
    FPCC_REQUIRE(A && W && out && m > 0, "linear_f16: bad arguments");
    int rc = f16_common(dtype, out_type, act, post_act, k, n, A, W, out);
    if (rc) return rc;
    TcArgs a = {};
    a.A = (const int8_t *)A; a.K = 2 * k; a.N = n;
    int tiles;
    if (sel_row) {
        FPCC_REQUIRE(sel_out && sel_offsets && n_groups > 0 && n_sel > 0, "linear_f16: incomplete selection");
        a.in_idx = sel_row; a.out_idx = sel_out; a.offsets = sel_offsets; a.n_groups = n_groups; a.n_pairs = n_sel; a.bias_per_group = 0;
        tiles = ceil_div(n_sel, TC_M) + n_groups;
    } else {
        a.n_groups = 1; a.n_pairs = m;
        tiles = ceil_div(m, TC_M);
        n_groups = 1;
    }
    FEpi fe = {bias, residual, slope, post_slope, act, post_act, out_type};
    EpiParams ep = {};
    if (dtype == 0) return launch_tc<1, 1>(a, W, (int64_t)n_groups * n, tiles, ep, fe, out, (cudaStream_t)stream);
    return launch_tc<1, 2>(a, W, (int64_t)n_groups * n, tiles, ep, fe, out, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// Weight gradient of the float sparse convolution on the tensor cores (training: SURVEY 8a row 19, the wgrad product of
// MinkowskiEngine's / torchsparse's backward, per kernel offset):
//     dW[k][ci][co] += sum over the pairs p of offset k of  X[in[p]][ci] * dY[out[p]][co]
// i.e. a GEMM whose CONTRACTION runs over the gathered rows.  Both operands are therefore MN-major for tcgen05 (idesc bits
// 15 / 16): a gathered row (one pair) is one K index and its channels are contiguous, so the rows the producers copy with
// cp.async land in shared memory exactly as the SWIZZLE_128B MN-major canonical layout wants them -- atoms of 8 rows x 128 B,
// the 64-channel atoms of an operand LBO = 8 KB apart, 8-row groups SBO = 1 KB apart -- no transpose anywhere.
// One tile = up to WG_CHUNK pairs of ONE offset (split-K); the fp32 accumulator [C_in (<= 2 x 128 lanes), C_out columns]
// lives in TMEM over the whole tile and is added into dW with red.global.add.f32 (partial sums of the tiles of an offset
// meet there, as in ME / torchsparse's atomics-based backward).
//   warps 0-3 gather producers, 4-7 epilogue (TMEM lane quarter = warp % 4), 8 TMEM owner + MMA issuer
// ---------------------------------------------------------------------------------------------
namespace fpcc {
constexpr int WG_PAIRS = 64;     // pairs per pipeline stage: four K = 16 instructions
constexpr int WG_CHUNK = 2048;   // pairs per tile
constexpr int WG_THREADS = 9 * 32;

struct WgArgs {
    const uint8_t *X, *dY;              // [*, c_in_p] / [*, c_out_p] fp16 or bf16 rows
    const int32_t *in_idx, *out_idx;    // compacted pair lists (fpcc_kmap_compact)
    const int4 *tiles;                  // per tile: (offset k, first pair, end pair, -)
    int n_tiles;
    int c_in_p, c_out_p;                // padded channels: c_in_p in {128, 256}, c_out_p a multiple of 64, <= 256
    int c_in, c_out;                    // real channels of dW [kvol, c_in, c_out]
    float *dW;
    int bf16, stages, tmem_cols;
};

__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);  // start address
    d |= (uint64_t)(8192u >> 4) << 16;             // leading byte offset: next 64-element atom along M / N
    d |= (uint64_t)(1024u >> 4) << 32;             // stride byte offset: next group of 8 K rows
    d |= (uint64_t)1 << 46;                        // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
    return d;
}

__global__ void __launch_bounds__(WG_THREADS, 1) wgrad_tc_kernel(WgArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int atoms_a = a.c_in_p / 64, atoms_b = a.c_out_p / 64;
    const int a_bytes = atoms_a * 8192, b_bytes = atoms_b * 8192, st_bytes = a_bytes + b_bytes;
    uint64_t *bars = (uint64_t *)(smem + (size_t)a.stages * st_bytes);
    uint64_t *full = bars, *empty = bars + 8, *tmem_full = bars + 16, *tmem_empty = bars + 17;
    uint32_t *tmem_ptr = (uint32_t *)(bars + 18);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ma = a.c_in_p / 128;

    if (warp == 8 && lane == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 128); mbar_init(&empty[s], 1); }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"((uint32_t)a.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp < 4) {
        // ---- gather producers: 8 consecutive lanes copy the 8 pieces of one 128-byte line (one pair, one 64-channel atom).
        // Line group g (16 of them) serves the pairs g, g+16, g+32, g+48 of a stage for every atom of both operands; their
        // 4 + 4 row indices are fetched one STAGE ahead into registers (a dependent index load per line serialised the
        // whole stage behind the L2 latency: 43 TFLOP/s for this kernel).
        const int grp = tid >> 3, piece = tid & 7;
        int it = 0;
        int32_t nx_in[4], nx_out[4];
        auto fetch_idx = [&](int t, int s) {
#pragma unroll
            for (int i = 0; i < 4; ++i) { nx_in[i] = -1; nx_out[i] = -1; }
            if (t >= a.n_tiles) return;
            const int4 tl = __ldg(&a.tiles[t]);
            const int base = tl.y + s * WG_PAIRS;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int p = base + grp + 16 * i;
                if (p < tl.z) { nx_in[i] = __ldg(&a.in_idx[p]); nx_out[i] = __ldg(&a.out_idx[p]); }
            }
        };
        fetch_idx(blockIdx.x, 0);
        for (int t = blockIdx.x; t < a.n_tiles; t += gridDim.x) {
            const int4 tl = __ldg(&a.tiles[t]);
            const int n_st = (tl.z - tl.y + WG_PAIRS - 1) / WG_PAIRS;
            // a tile of no pairs consumes none of the indices fetched for it: fetch the next tile's here, or that tile's
            // first stage would gather nothing
            if (n_st <= 0) fetch_idx(t + gridDim.x, 0);
            for (int s = 0; s < n_st; ++s, ++it) {
                int32_t cin_[4], cout_[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { cin_[i] = nx_in[i]; cout_[i] = nx_out[i]; }
                if (s + 1 < n_st) fetch_idx(t, s + 1);
                else fetch_idx(t + gridDim.x, 0);
                const int stage = it % a.stages;
                mbar_wait(&empty[stage], ((it / a.stages) & 1) ^ 1);
                const uint32_t sA = smem_u32(smem + (size_t)stage * st_bytes), sB = sA + a_bytes;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int kk = grp + 16 * i;  // K row of the stage = pair
                    const uint32_t sw = (uint32_t)((piece ^ (kk & 7)) << 4) + (uint32_t)kk * 128;
                    const bool ok = cin_[i] >= 0;
                    const uint8_t *xa = a.X + (int64_t)(ok ? cin_[i] : 0) * a.c_in_p * 2 + piece * 16;
                    const uint8_t *ya = a.dY + (int64_t)(ok ? cout_[i] : 0) * a.c_out_p * 2 + piece * 16;
                    for (int at = 0; at < atoms_a; ++at) cp_async16(sA + at * 8192 + sw, xa + at * 128, ok ? 16u : 0u);
                    for (int at = 0; at < atoms_b; ++at) cp_async16(sB + at * 8192 + sw, ya + at * 128, ok ? 16u : 0u);
                }
                asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&full[stage])) : "memory");
            }
        }
    } else if (warp == 8) {
        // ---- MMA issuer
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | ((uint32_t)a.bf16 << 7) | ((uint32_t)a.bf16 << 10) | (1u << 15) | (1u << 16) |
                                   ((uint32_t)(a.c_out_p >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            int it = 0, j = 0;
            for (int t = blockIdx.x; t < a.n_tiles; t += gridDim.x, ++j) {
                const int4 tl = __ldg(&a.tiles[t]);
                const int n_st = (tl.z - tl.y + WG_PAIRS - 1) / WG_PAIRS;
                mbar_wait(tmem_empty, (j & 1) ^ 1);  // the epilogue has drained the previous tile's accumulator
                tc_fence_after();
                for (int s = 0; s < n_st; ++s, ++it) {
                    const int stage = it % a.stages;
                    mbar_wait(&full[stage], (it / a.stages) & 1);
                    fence_proxy_async();
                    tc_fence_after();
                    const uint32_t sA = smem_u32(smem + (size_t)stage * st_bytes), sB = sA + a_bytes;
#pragma unroll
                    for (int q = 0; q < WG_PAIRS / 16; ++q) {  // 16 pairs (K) per instruction: 16 rows of 128 B
                        const uint64_t bd = umma_desc_mn_sw128(sB + q * 2048);
                        for (int mb = 0; mb < ma; ++mb)
                            umma_f16(tmem_base + (uint32_t)(mb * a.c_out_p), umma_desc_mn_sw128(sA + mb * 16384 + q * 2048), bd, idesc,
                                     (uint32_t)(s > 0 || q > 0));
                    }
                    umma_commit(&empty[stage]);
                }
                if (n_st > 0) umma_commit(tmem_full);
                else mbar_arrive(tmem_full);
            }
        }
    } else {
        // ---- epilogue: accumulator rows = input channels (TMEM lanes), columns = output channels
        const int quarter = warp & 3;
        int j = 0;
        for (int t = blockIdx.x; t < a.n_tiles; t += gridDim.x, ++j) {
            const int4 tl = __ldg(&a.tiles[t]);
            mbar_wait(tmem_full, j & 1);
            tc_fence_after();
            if (tl.z > tl.y) {
                for (int mb = 0; mb < ma; ++mb) {
                    const int ci = mb * 128 + quarter * 32 + lane;
                    float *drow = a.dW + ((int64_t)tl.x * a.c_in + ci) * a.c_out;
                    for (int c0 = 0; c0 < a.c_out_p; c0 += 16) {
                        uint32_t v[16];
                        __syncwarp();
                        tmem_ld16(tmem_base + (uint32_t)(mb * a.c_out_p + c0) + ((uint32_t)(quarter * 32) << 16), v);
                        if (ci < a.c_in) {
                            if ((a.c_out & 3) == 0) {  // 16-byte aligned rows: four columns per reduction
#pragma unroll
                                for (int q = 0; q < 16; q += 4)
                                    if (c0 + q < a.c_out)
                                        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(drow + c0 + q), "f"(__uint_as_float(v[q])),
                                                     "f"(__uint_as_float(v[q + 1])), "f"(__uint_as_float(v[q + 2])), "f"(__uint_as_float(v[q + 3])) : "memory");
                            } else {
#pragma unroll
                                for (int q = 0; q < 16; ++q)
                                    if (c0 + q < a.c_out) atomicAdd(drow + c0 + q, __uint_as_float(v[q]));
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tmem_empty);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)a.tmem_cols) : "memory");
    }
}
}  // namespace fpcc

extern "C" int fpcc_spconv_wgrad_f16(const void *x, const void *dy, int dtype, int c_in_p, int c_out_p, const int32_t *in_idx,
                                     const int32_t *out_idx, const int32_t *tiles, int n_tiles, float *dw, int c_in, int c_out,
                                     void *stream) {
    using namespace fpcc;
    FPCC_REQUIRE(x && dy && in_idx && out_idx && tiles && dw, "spconv_wgrad_f16: NULL pointer");
    FPCC_REQUIRE(dtype == 0 || dtype == 1, "spconv_wgrad_f16: dtype 0 (fp16) or 1 (bf16)");
    FPCC_REQUIRE((c_in_p == 128 || c_in_p == 256) && c_out_p % 64 == 0 && c_out_p >= 64 && c_out_p <= 256,
                 "spconv_wgrad_f16: padded channels must be C_in in {128, 256}, C_out a multiple of 64 up to 256 (got %d, %d)", c_in_p, c_out_p);
    FPCC_REQUIRE(c_in > 0 && c_in <= c_in_p && c_out > 0 && c_out <= c_out_p, "spconv_wgrad_f16: real channels exceed the padded ones");
    FPCC_REQUIRE((((uintptr_t)x | (uintptr_t)dy) & 15) == 0, "spconv_wgrad_f16: rows must be 16-byte aligned");
    if (n_tiles <= 0) return FPCC_OK;
    WgArgs a;
    a.X = (const uint8_t *)x; a.dY = (const uint8_t *)dy; a.in_idx = in_idx; a.out_idx = out_idx; a.tiles = (const int4 *)tiles;
    a.n_tiles = n_tiles; a.c_in_p = c_in_p; a.c_out_p = c_out_p; a.c_in = c_in; a.c_out = c_out; a.dW = dw; a.bf16 = dtype;
    const int st_bytes = (c_in_p / 64 + c_out_p / 64) * 8192;
    a.stages = (int)((200 * 1024) / st_bytes);
    if (a.stages > 6) a.stages = 6;
    int cols = (c_in_p / 128) * c_out_p, pow2 = 32;
    while (pow2 < cols) pow2 <<= 1;
    a.tmem_cols = pow2;
    const size_t smem = 1024 + (size_t)a.stages * st_bytes + 256;
    static bool configured = false;
    if (!configured) {
        FPCC_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        configured = true;
    }
    int sms = g_sm_budget > 0 && g_sm_budget < sm_count() ? g_sm_budget : sm_count();
    const int grid = n_tiles < sms ? n_tiles : sms;
    wgrad_tc_kernel<<<grid, WG_THREADS, smem, (cudaStream_t)stream>>>(a);
    FPCC_LAUNCH_CHECK();
    return FPCC_OK;
}

extern "C" int fpcc_mma_i8_peak(int iters, int n, double *tops_out, void *stream) {
    using namespace fpcc;
    FPCC_REQUIRE(iters > 0 && tops_out && n >= 16 && n <= 256 && n % 16 == 0, "mma_i8_peak: bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    size_t smem = 1024 + TC_M * TC_KB + 256 * TC_KB;
    FPCC_CUDA(cudaFuncSetAttribute(mma_i8_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEvent_t e0, e1;
    FPCC_CUDA(cudaEventCreate(&e0));
    FPCC_CUDA(cudaEventCreate(&e1));
    int sms = sm_count();
    mma_i8_peak_kernel<<<sms, 128, smem, s>>>(iters / 8 + 1, n);  // warm-up
    FPCC_CUDA(cudaEventRecord(e0, s));
    mma_i8_peak_kernel<<<sms, 128, smem, s>>>(iters, n);
    FPCC_CUDA(cudaEventRecord(e1, s));
    FPCC_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    FPCC_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tops_out = 2.0 * TC_M * n * 32.0 * 4.0 * iters * sms / (ms * 1e-3) / 1e12;
    return FPCC_OK;
}

#ifdef FPCC_TC_TRACE
extern "C" int fpcc_trace_read(unsigned long long *host, int n) {
    FPCC_CUDA(cudaDeviceSynchronize());
    FPCC_CUDA(cudaMemcpyFromSymbol(host, fpcc::g_trace, sizeof(unsigned long long) * 8 * (size_t)n));
    return FPCC_OK;
}
#endif

extern "C" int fpcc_gemm_engine(int k, int n, int kvol, int has_zp_comp) {
    return fpcc::tc_enabled() && !has_zp_comp && k >= 32 && k % 16 == 0 && n >= 16 && kvol <= fpcc::TC_MAX_KVOL;
}

extern "C" int fpcc_set_sm_budget(int sms) {
    fpcc::g_sm_budget = sms > 0 ? sms : 0;
    return FPCC_OK;
}

extern "C" int fpcc_set_tc_mode(int mode) {
    fpcc::g_tc_mode = mode ? 1 : 0;
    return FPCC_OK;
}
