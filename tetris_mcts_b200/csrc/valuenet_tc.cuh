// valuenet_tc.cuh — the reference value network (model/model_vv.py:13-52) on Blackwell tensor cores (sm_100a).
//
// Precision: north_star asks value outputs within 1e-5 of the reference's fp32.  Plain bf16/tf32/fp16 MMAs cannot
// reach that, so every fp32 operand x is split into two fp16 terms x = x1 + x2 (11 + 11 = 22 mantissa bits, the
// precision class of 3xTF32) and each product a*b is accumulated in fp32 (TMEM) as a1*b2 + a2*b1 + a1*b1 (the dropped
// a2*b2 is < 2^-22 relative).  Operands are pre-scaled by exact powers of two (activations x16, weights x64) so that the
// low terms stay in fp16's normal range; the epilogues undo the 2^10.  Three fp16 MMAs replace one fp32 product.
//
//   k_tc_conv  one persistent CTA per SM, four boards in flight (software pipeline):
//              obs key -> im2col (exact fp16) -> conv1 as one K=16 MMA per M tile -> epilogue (bias, ReLU, split) -> smem
//              conv2 / conv3 as shift-GEMMs: activations live in shared memory channel-chunk-major
//              ([8-channel chunk][pixel row][16 B]) on an 8-wide pixel grid, so the A operand of filter row dy is the SAME
//              array started dy*8 rows later — a canonical no-swizzle K-major UMMA layout with SBO = 128 B,
//              LBO = rows*16 B; the three horizontal taps are stacked along N (N = 96) and summed by the epilogue with
//              two lane shuffles.  tcgen05.mma (M=128 pixels, K=16) issued by one thread, accumulators in TMEM,
//              completion through tcgen05.commit -> mbarrier; epilogues read TMEM with tcgen05.ld, apply bias+ReLU,
//              re-split (fp16 x2) and write the next layer's operand (or act3 to HBM in the FC kernel's tile layout).
//   k_tc_fc    [R,1792] x [1792,256] on the FC pipeline it shares with k_tdc_fc (fc_pipeline below: 128-row tiles, operands
//              streamed by cp.async.bulk (1-D TMA) into an 8-stage mbarrier ring — both operands are stored in HBM already in the
//              canonical UMMA layout, so one bulk copy per operand block needs no tensor map; producer / MMA issuer / 4 epilogue
//              warps); its epilogue fuses bias+ReLU+fc_out+sigmoid+affine and scatters (v, var) to the requesting tree slot.
#pragma once
#include <cuda_fp16.h>
#include "search_dev.cuh"
#include "valuenet_simt.cuh"

namespace b200 {

// ---------------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// whole warp waits, one lane polls (32 lanes polling the same word is shared-memory traffic the MMA operand fetch competes with)
__device__ __forceinline__ void mbar_wait_warp(uint64_t *bar, uint32_t parity);
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0u;
}
__device__ __forceinline__ void mbar_wait_warp(uint64_t *bar, uint32_t parity) {
    // most waits of the conv pipeline find their phase already complete: one warp-wide test_wait (a broadcast read) answers that
    // without the lane-0 poll + __syncwarp round trip
    if (__all_sync(0xffffffffu, mbar_test(bar, parity))) return;
    if ((threadIdx.x & 31) == 0) mbar_wait(bar, parity);
    __syncwarp();
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {   // 1-D TMA (UBLKCP)
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem) {   // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {   // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}

// K-major, no-swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, version 1):
// rows of a core matrix are 16 B apart, 8-row groups SBO apart, the two 16-byte K chunks LBO apart.
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
// kind::f16 instruction descriptor: D=f32 (bits 4-5 = 1), A=B=fp16 (format 0), both K-major, N>>3 at bit 17, M>>4 at bit 24
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
constexpr float TC_SCALE_A = 16.f, TC_SCALE_W = 64.f, TC_UNSCALE = 1.f / 1024.f;
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {   // lane i of the warp <- TMEM lane (quadrant*32 + i), 16 columns
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8_sum2(uint32_t taddr, float (&v)[8]) {
    float w1[8], w2[8];
    tmem_ld8(taddr + 32, w2);
    tmem_ld8(taddr, w1);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = (w2[i] + w1[i]) * TC_UNSCALE;
}

// accumulator blocks a*W1 | a*W2 sit 32 columns apart: add the small one first, undo the operand scaling
__device__ __forceinline__ void tmem_ld16_sum2(uint32_t taddr, float (&v)[16]) {
    float w1[16], w2[16];
    tmem_ld16(taddr + 32, w2);
    tmem_ld16(taddr, w1);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = (w2[i] + w1[i]) * TC_UNSCALE;
}

// x = x1 + x2 with fp16 terms (round-to-nearest each step); eight fp32 values -> two 16-byte chunks (one per split)
__device__ __forceinline__ void split8(const float (&x)[8], uint4 &c1, uint4 &c2) {
    uint32_t a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __half2 h = __floats2half2_rn(x[2 * i], x[2 * i + 1]);                 // one packed conversion per pair
        const float2 f = __half22float2(h);
        const __half2 l = __floats2half2_rn(x[2 * i] - f.x, x[2 * i + 1] - f.y);
        a[i] = *reinterpret_cast<const uint32_t *>(&h); b[i] = *reinterpret_cast<const uint32_t *>(&l);
    }
    c1 = make_uint4(a[0], a[1], a[2], a[3]);
    c2 = make_uint4(b[0], b[1], b[2], b[3]);
}

// ---------------------------------------------------------------------------------------------------- conv kernel
// Measured on B200 (scripts/probe/mma_probe.cu): a tcgen05.mma costs max(44.7, ~N/2) clk however small it is, so the
// layers are cut into FEW, WIDE instructions.  The three horizontal taps (dx) of a 3x3 filter are stacked along N:
//   D'[p][dx*32 + cout] = sum_{dy, cin} act[p + dy*8][cin] * W[dy][dx][cin][cout]          (A operand shifted by dy*8 rows only)
//   out[p][cout]        = D'[p][0*32+cout] + D'[p+1][1*32+cout] + D'[p+2][2*32+cout]        (epilogue: two lane shuffles)
// All three layers live on an 8-wide pixel grid (p = y*8 + x), so p+dx never leaves the 32-lane warp that owns the row.
// 18 MMAs (3 dy x 2 channel halves x 3 split products, N = 96) replace the 36 narrow ones of the tap-by-tap form, and
// conv1 (K = 9 taps, exact {-1,0,1} inputs) runs on the tensor core too from an im2col operand the workers build.
// (Two independent worker sets of 8 warps x 16 channels on alternating boards, one MMA issuer each, were measured on B200 at 3 204 clk per
// board against 2 751 with one set — profiles/exp_variants_r2f.txt — and removed.)
constexpr int TCC_WORKERS = 512;            // warps 0-15: the three epilogues
constexpr int TCC_ISSUER = TCC_WORKERS / 32; // warp 16: MMA issuer of conv1 + conv2 (one elected lane)
constexpr int TCC_ISSUER3 = TCC_ISSUER + 1; // warp 17: MMA issuer of conv3.  A 56-clk MMA costs its issuing thread ~8 dependent instructions
                                            // (uniform-register moves + the elect loop) and that thread shares its scheduler with four busy
                                            // worker warps: one issuer alone cannot keep the tensor pipe fed, two (on two schedulers) can.
constexpr int TCC_LOADER = TCC_ISSUER + 2;  // warp 18: fetches the observation keys of the CTA's boards into a shared-memory ring
constexpr int TCC_THREADS = TCC_WORKERS + 96;
constexpr int TCC_R = 144;                  // activation rows per board: 18x8 grid (act1) / 16x8 grid + the dy shifts (act2)
constexpr int TCC_WBLOCK = 2 * 2 * 96 * 16;  // one (dy, channel half) block: [weight split 2][chunk 2][n = dx*32 + cout][16 B]
constexpr int TCC_WBYTES = 6 * TCC_WBLOCK;   // one conv layer = 36864 B
constexpr int TCC_W1BYTES = 2 * 64 * 16;     // conv1: [chunk 2][n = split*32 + cout][16 B], k = tap (9 of 16 used)
constexpr int TCC_SLOTS = 4;                // boards in flight (barrier rings, im2col operands)
constexpr int TCC_KEYS_AHEAD = 4;           // observation keys the loader warp keeps in flight (registers)
constexpr int TCC_RUN = 4;                  // consecutive requests handed to a CTA at a time (a power of two)
constexpr int TCC_ASLOT = 2 * 4 * TCC_R * 16;    // operand buffer of one board: act1 [split][chunk 4][144 rows][16 B]
constexpr int TCC_IMROWS = 256;             // im2col rows per board: 144 used, two M=128 tiles
constexpr int TCC_IMSLOT = 2 * TCC_IMROWS * 16;  // [chunk 2][256 rows][16 B] fp16
// act2 overwrites the slot's act1 in place (conv2 has finished reading by then), and a slot's three accumulators reuse the same 128 TMEM
// columns in turn: board i of a CTA lives in slot i % TCC_SLOTS throughout.
constexpr int TCC_OFF_W2 = 0;
constexpr int TCC_OFF_W3 = TCC_OFF_W2 + TCC_WBYTES;
constexpr int TCC_OFF_W1 = TCC_OFF_W3 + TCC_WBYTES;
constexpr int TCC_OFF_A1 = TCC_OFF_W1 + TCC_W1BYTES;
constexpr int TCC_OFF_IM = TCC_OFF_A1 + TCC_SLOTS * TCC_ASLOT;
constexpr int TCC_OFF_BIAS = TCC_OFF_IM + TCC_SLOTS * TCC_IMSLOT;   // 96 floats
constexpr int TCC_OFF_KEY = TCC_OFF_BIAS + 96 * 4;                  // TCC_SLOTS x 32 words: the front-end warp's row table (20 rows: settled | piece << 16)
constexpr int TCC_OFF_BAR = TCC_OFF_KEY + TCC_SLOTS * 32 * 4;       // 6 x TCC_SLOTS mbarriers + tmem pointer
constexpr int TCC_SMEM = TCC_OFF_BAR + 6 * TCC_SLOTS * 8 + 16;
constexpr int TCC_TMEM_COLS = 512;
constexpr int ACT3_KCHUNKS = 224;           // 1792 / 8
static_assert(TCC_SMEM <= 227 * 1024, "k_tc_conv shared memory");

struct TcWeights {
    const uint8_t *wc1;         // TCC_W1BYTES
    const uint8_t *wc2, *wc3;   // TCC_WBYTES each, already in the shared-memory layout
    const uint8_t *wfc;         // [split 2][k16 block 112][chunk 2][n 256][16 B]
};

// act3 in HBM, FC-tile layout: [split][tile of 128 rows][k chunk 224][row 128][8 fp16], k' = (y*4 + x)*32 + c
__device__ __forceinline__ size_t act3_off(int split, int n_tiles, int ridx, int kchunk) {
    return ((((size_t)split * n_tiles + (ridx >> 7)) * ACT3_KCHUNKS + kchunk) * 128 + (ridx & 127)) * 16;
}

// three 8-column accumulator slices (32 columns apart) of this thread's TMEM lane, one wait
__device__ __forceinline__ void tmem_ld8x3(uint32_t taddr, float (&a)[8], float (&b)[8], float (&c)[8]) {
    uint32_t r[24];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%24];\n"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%8,%9,%10,%11,%12,%13,%14,%15}, [%25];\n"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%16,%17,%18,%19,%20,%21,%22,%23}, [%26];\n"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23])
        : "r"(taddr), "r"(taddr + 32), "r"(taddr + 64)
        : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) { a[i] = __uint_as_float(r[i]); b[i] = __uint_as_float(r[8 + i]); c[i] = __uint_as_float(r[16 + i]); }
}

// two 8-column accumulator slices (32 columns apart), one wait
__device__ __forceinline__ void tmem_ld8x2(uint32_t taddr, float (&a)[8], float (&b)[8]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%16];\n"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%8,%9,%10,%11,%12,%13,%14,%15}, [%17];\n"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr), "r"(taddr + 32)
        : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) { a[i] = __uint_as_float(r[i]); b[i] = __uint_as_float(r[8 + i]); }
}

// out[p] = D'[p][dx=0] + D'[p+1][dx=1] + D'[p+2][dx=2] for the 8 couts of this warp's chunk (see the header of this section)
__device__ __forceinline__ void tmem_ld_conv_sum(uint32_t taddr, float (&v)[8]) {
    float d0[8], d1[8], d2[8];
    tmem_ld8x3(taddr, d0, d1, d2);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const float s1 = __shfl_down_sync(0xffffffffu, d1[e], 1), s2 = __shfl_down_sync(0xffffffffu, d2[e], 2);
        v[e] = (s2 + s1) + d0[e];          // still carries the operand scaling 2^10: the callers fold TC_UNSCALE into their bias fma
    }
}

// One 3x3 layer = 18 tcgen05.mma of N = 96: for each (dy, channel half): a1*W1, a1*W2, a2*W1 into the same 96 columns.
__device__ __forceinline__ void issue_conv_layer(uint32_t tmem_d, uint32_t a_addr, uint32_t w_addr) {
    const uint64_t a0 = umma_desc(a_addr, TCC_R * 16, 128), b0 = umma_desc(w_addr, 96 * 16, 128);
    constexpr uint32_t idesc = umma_idesc_f16(128, 96);
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t a_hi = 2 * h * TCC_R + dy * 8, a_lo = a_hi + 4 * TCC_R;          // 16-byte units
            const uint32_t b_hi = (dy * 2 + h) * (TCC_WBLOCK / 16), b_lo = b_hi + 2 * 96;
            umma_f16(tmem_d, a0 + a_hi, b0 + b_hi, idesc, (dy | h) ? 1u : 0u);
            umma_f16(tmem_d, a0 + a_hi, b0 + b_lo, idesc, 1u);
            umma_f16(tmem_d, a0 + a_lo, b0 + b_hi, idesc, 1u);
        }
    }
}


__global__ void __launch_bounds__(TCC_THREADS, 1)
k_tc_conv(NetWeights W, TcWeights TW, const uint2 *req, const int32_t *n_req_ptr, const uint32_t *keys, int M, uint8_t *act3,
          int n_tiles, unsigned long long *prof) {
#define PROF_T(i) do { if (prof && do_prof) { long long _n = clock64(); pacc[i] += _n - ptick; ptick = _n; } } while (0)
    extern __shared__ __align__(128) uint8_t smem[];
    float *sB = reinterpret_cast<float *>(smem + TCC_OFF_BIAS);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + TCC_OFF_BAR);
    constexpr int NS = TCC_SLOTS;
    uint64_t *bar_c1 = bars, *bar_c2 = bars + NS, *bar_c3 = bars + 2 * NS;             // tensor core -> workers: layer of slot done
    uint64_t *bar_a0 = bars + 3 * NS, *bar_a1 = bars + 4 * NS, *bar_a2 = bars + 5 * NS; // workers -> issuer: operand of slot written
    uint32_t *sKey = reinterpret_cast<uint32_t *>(smem + TCC_OFF_KEY);
    uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(smem + TCC_OFF_BAR + 6 * NS * 8);
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    // ---- one-time setup: weights into smem, zeroed operands, barriers, TMEM
    for (int i = t; i < TCC_WBYTES / 16; i += TCC_THREADS) {
        reinterpret_cast<uint4 *>(smem + TCC_OFF_W2)[i] = reinterpret_cast<const uint4 *>(TW.wc2)[i];
        reinterpret_cast<uint4 *>(smem + TCC_OFF_W3)[i] = reinterpret_cast<const uint4 *>(TW.wc3)[i];
    }
    for (int i = t; i < TCC_W1BYTES / 16; i += TCC_THREADS) reinterpret_cast<uint4 *>(smem + TCC_OFF_W1)[i] = reinterpret_cast<const uint4 *>(TW.wc1)[i];
    for (int i = t; i < (TCC_OFF_BIAS - TCC_OFF_A1) / 16; i += TCC_THREADS) reinterpret_cast<uint4 *>(smem + TCC_OFF_A1)[i] = make_uint4(0, 0, 0, 0);
    if (t < 32) { sB[t] = W.b1[t]; sB[32 + t] = W.b2[t]; sB[64 + t] = W.b3[t]; }
    if (t == 0) {
        for (int i = 0; i < 3 * NS; ++i) mbar_init(&bars[i], 1);
        for (int i = 3 * NS; i < 4 * NS; ++i) mbar_init(&bars[i], 1);                      // a0: the front-end warp alone builds the conv1 operand
        for (int i = 4 * NS; i < 6 * NS; ++i) mbar_init(&bars[i], TCC_WORKERS / 32);   // a1, a2: one arrival per worker warp
        fence_barrier_init();
    }
    if (warp == TCC_ISSUER) tmem_alloc<TCC_TMEM_COLS>(tmem_ptr);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const int n_req = *n_req_ptr;
    // Boards are handed out in runs of TCC_RUN consecutive requests (neighbouring act3 rows get written close in time; short runs keep
    // the CTAs' board counts within TCC_RUN of each other: with runs of 8 the last CTAs had 4 % more work); board i of
    // this CTA's sequence lives in slot i % 4.  Four boards are in flight at different stages (software pipeline):
    //   workers, iteration i :  S0(i) im2col | E2(i-2) conv2 epilogue | E3(i-3) conv3 epilogue | E1(i) conv1 epilogue
    //   issuer,  iteration i :  conv2(i-1) | conv1(i) | conv3(i-2), each as soon as the workers have written its operand
    // The order is chosen so that the tensor pipe never runs dry: conv2(i-1)'s operand was finished at the end of the
    // previous iteration (E1 comes last), conv1(i) is short and queued behind it, conv3(i-2)'s operand (E2) is ready long
    // before conv2 retires; the workers drain older boards (E2, E3) while conv2 runs and reach E1(i) after conv1(i) is done.
    const int n_runs = (n_req + TCC_RUN - 1) / TCC_RUN;
    int n_local = 0;
    for (int run = blockIdx.x; run < n_runs; run += gridDim.x) n_local += min(TCC_RUN, n_req - run * TCC_RUN);
    auto board_of = [&](int i) -> int { return ((i / TCC_RUN) * (int)gridDim.x + (int)blockIdx.x) * TCC_RUN + (i % TCC_RUN); };
    if (warp == TCC_ISSUER) {
        // ===================================================== MMA issuer
        if (lane == 0) {
            const uint32_t s_w1 = smem_u32(smem + TCC_OFF_W1), s_w2 = smem_u32(smem + TCC_OFF_W2), s_w3 = smem_u32(smem + TCC_OFF_W3);
            const uint32_t s_act = smem_u32(smem + TCC_OFF_A1), s_im = smem_u32(smem + TCC_OFF_IM);
            const bool do_prof = blockIdx.x == 0;
            long long pacc[16] = {0}, ptick = clock64();
            for (int i = 0; i < n_local + 1; ++i) {
                // conv1(i) goes FIRST: its operand comes from the front-end warp (boards ahead), its accumulator columns were last read by
                // E3(i-4), and E1(i-1) — the last phase of the workers' previous iteration, a1(i-1) — implies that E3(i-4) is done.  With
                // conv1 queued behind the 18 MMAs of conv2 (round 1: the workers built the operand, so it could not be ready earlier) the
                // workers stood at E1(i) for ~1 k clk per board waiting for it.
                if (i >= 1) {
                    const int j = i - 1, slot = j % NS;
                    mbar_wait(&bar_a1[slot], (uint32_t)(j / NS) & 1u);
                    PROF_T(10);
                }
                if (i < n_local) {                               // conv1 (model_vv.py:32): im2col [256 x 16] x W1 [16 x 64], two M tiles
                    const int slot = i % NS;
                    mbar_wait(&bar_a0[slot], (uint32_t)(i / NS) & 1u);
                    PROF_T(8);
                    tc_fence_after();
                    const uint64_t a0 = umma_desc(s_im + slot * TCC_IMSLOT, TCC_IMROWS * 16, 128), b0 = umma_desc(s_w1, 64 * 16, 128);
                    umma_f16(tmem_base + slot * 128, a0, b0, umma_idesc_f16(128, 64), 0u);
                    umma_f16(tmem_base + slot * 128 + 64, a0 + 128, b0, umma_idesc_f16(128, 64), 0u);
                    umma_commit(&bar_c1[slot]);
                    PROF_T(9);
                }
                if (i >= 1) {                                    // conv2 (model_vv.py:34): act1 on the 18x8 grid
                    const int j = i - 1, slot = j % NS;
                    tc_fence_after();
                    issue_conv_layer(tmem_base + slot * 128, s_act + slot * TCC_ASLOT, s_w2);
                    umma_commit(&bar_c2[slot]);
                    PROF_T(11);
                }
            }
            if (prof && do_prof) for (int i = 8; i < 12; ++i) atomicAdd(&prof[i], (unsigned long long)pacc[i]);
        }
    } else if (warp == TCC_ISSUER3) {
        // ===================================================== second MMA issuer: conv3 (model_vv.py:36)
        if (lane == 0) {
            const uint32_t s_w3 = smem_u32(smem + TCC_OFF_W3);
            const bool do_prof = blockIdx.x == 0;
            long long pacc[16] = {0}, ptick = clock64();
            const uint32_t s_act = smem_u32(smem + TCC_OFF_A1);
            for (int j = 0; j < n_local; ++j) {                  // act2 on the 16x8 grid
                const int slot = j % NS;
                mbar_wait(&bar_a2[slot], (uint32_t)(j / NS) & 1u);
                PROF_T(12);
                tc_fence_after();
                issue_conv_layer(tmem_base + slot * 128, s_act + slot * TCC_ASLOT, s_w3);
                umma_commit(&bar_c3[slot]);
                PROF_T(13);
            }
            if (prof && do_prof) for (int i = 12; i < 14; ++i) atomicAdd(&prof[i], (unsigned long long)pacc[i]);
        }
    } else if (warp == TCC_LOADER) {
        // ===================================================== front end (one warp): observation key -> conv1 operand.
        // A key is a random 48-byte read from an arena of tens of GB (~2.4 k clk); TCC_KEYS_AHEAD of them are kept in flight.  The same
        // warp then builds the im2col operand of conv1 (fp16, exact {-1,0,1}): row p = y*8 + x of the 18x8 output grid, k = tap = dy*3 + dx,
        // taps 0..7 as ONE 16-byte store, tap 8 in the second k chunk.  (Round 1 had all 16 worker warps build it, 27 % of their cycle;
        // one warp running up to TCC_SLOTS boards ahead of the epilogues does it off the workers' critical path.)
        uint2 rqs = make_uint2(0, 0);
        uint32_t kq[TCC_KEYS_AHEAD];
        auto fetch = [&](int i) -> uint32_t {                       // whole warp; board i of this CTA (i < n_local)
            if ((i & 31) == 0 && i + lane < n_local) rqs = req[board_of(i + lane)];
            const uint32_t gx = __shfl_sync(0xffffffffu, rqs.x, i & 31), gy = __shfl_sync(0xffffffffu, rqs.y, i & 31);
            return lane < 12 ? keys[((size_t)gx * M + (gy & 0x0fffffffu)) * KEY_WORDS + lane] : 0u;
        };
#pragma unroll
        for (int j = 0; j < TCC_KEYS_AHEAD; ++j) kq[j] = j < n_local ? fetch(j) : 0u;
        for (int i0 = 0; i0 < n_local; i0 += TCC_KEYS_AHEAD) {
#pragma unroll
            for (int j = 0; j < TCC_KEYS_AHEAD; ++j) {
                const int i = i0 + j;
                if (i >= n_local) break;
                const int slot = i % NS;
                // row table: lane r < 20 holds board row r: settled cells in bits 0..9, the falling piece's cells in bits 16..25
                const uint32_t kw = kq[j];
                const uint32_t rowpair = __shfl_sync(0xffffffffu, kw, (lane >> 1) & 15), pcs = __shfl_sync(0xffffffffu, kw, 10);
                uint32_t tab = (rowpair >> ((lane & 1) * 16)) & 0x3ffu;
#pragma unroll
                for (int k = 0; k < 4; ++k) {                    // the falling piece's cells (sorted bytes of key word 10)
                    const uint32_t cell = (pcs >> (8 * k)) & 0xffu, pr = (cell * 205u) >> 11, pcol = cell - pr * 10u;
                    tab |= (pr == (uint32_t)lane ? 1u : 0u) << (16 + pcol);
                }
                if (i + TCC_KEYS_AHEAD < n_local) kq[j] = fetch(i + TCC_KEYS_AHEAD);            // next key of this register, in flight while the operand is built
                if (i >= NS) mbar_wait_warp(&bar_c1[slot], (uint32_t)((i - NS) / NS) & 1u);     // conv1 of the slot's previous board has read its operand
                if (lane < 20) sKey[slot * 32 + lane] = tab;
                __syncwarp();
                uint8_t *im = smem + TCC_OFF_IM + slot * TCC_IMSLOT;
#pragma unroll
                for (int pp = 0; pp < 5; ++pp) {                 // 144 pixels over 32 lanes
                    const int p = pp * 32 + lane;
                    if (p < 144) {
                        const int y = p >> 3, x = p & 7;
                        uint32_t hv[9];
#pragma unroll
                        for (int dy = 0; dy < 3; ++dy) {
                            const uint32_t rw = sKey[slot * 32 + y + dy] >> x;
#pragma unroll
                            for (int dx = 0; dx < 3; ++dx)       // 1 settled, -1 falling piece, 0 empty (model_vv.py:212)
                                hv[dy * 3 + dx] = ((rw >> dx) & 1u) * 0x3C00u | ((rw >> (16 + dx)) & 1u) * 0xBC00u;
                        }
                        *reinterpret_cast<uint4 *>(im + p * 16) =
                            make_uint4(hv[0] | (hv[1] << 16), hv[2] | (hv[3] << 16), hv[4] | (hv[5] << 16), hv[6] | (hv[7] << 16));   // taps 0..7
                        *reinterpret_cast<uint32_t *>(im + TCC_IMROWS * 16 + p * 16) = hv[8];                                        // tap 8
                    }
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_a0[slot]);
            }
        }
    } else {
        // ===================================================== workers (512 threads)
        const bool do_prof = blockIdx.x == 0 && t == 0;
        long long pacc[16] = {0}, ptick = clock64();
        const int q = warp & 3, cq = warp >> 2, m = q * 32 + lane;       // TMEM lane quadrant, 8-cout chunk, pixel row
        const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + cq * 8;
        // this warp's 8 couts, all three layers.  relu(x * 2^-10 + b) * 16 == relu(fma(x, 2^-6, 16 b)) bit for bit (scaling by a power of two commutes
        // with rounding): the biases are kept pre-scaled and an epilogue value costs one fma + one max instead of mul, add, max, mul
        float bias1[8], bias2[8], bias3[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) { bias1[e] = sB[cq * 8 + e] * TC_SCALE_A; bias2[e] = sB[32 + cq * 8 + e] * TC_SCALE_A; bias3[e] = sB[64 + cq * 8 + e] * TC_SCALE_A; }
        constexpr float K23 = TC_UNSCALE * TC_SCALE_A, K1 = TC_SCALE_A / TC_SCALE_W;
        const int n_iter = n_local + 3;
        auto phase_e2 = [&](int i) {
            // ---- E2(i-2): conv2 epilogue: dx sum + bias + ReLU + split -> act2
            if (i >= 2 && i - 2 < n_local) {
                const int j = i - 2, slot = j % NS;
                mbar_wait_warp(&bar_c2[slot], (uint32_t)(j / NS) & 1u);
                PROF_T(3);
                tc_fence_after();
                float v[8];
                tmem_ld_conv_sum(t_lane + slot * 128, v);
                {
                    float o[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[e] = fmaxf(fmaf(v[e], K23, bias2[e]), 0.f);
                    uint4 c1, c2;
                    split8(o, c1, c2);
                    if ((m & 7) < 6) {                           // 16x8 grid, in place of the slot's act1
                        uint8_t *base = smem + TCC_OFF_A1 + slot * TCC_ASLOT + (cq * TCC_R + m) * 16;
                        *reinterpret_cast<uint4 *>(base) = c1;
                        *reinterpret_cast<uint4 *>(base + 4 * TCC_R * 16) = c2;
                    }
                }
                tc_fence_before();
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_a2[slot]);     // 32 same-address arrivals would serialise in the shared-memory pipe the MMAs read through
                PROF_T(4);
            }
        };
        auto phase_e3 = [&](int i) {
            // ---- E3: conv3 epilogue: tap sum + bias + ReLU + split -> act3 in HBM (FC tile layout)
            if (i >= 3) {
                const int j = i - 3, slot = j % NS, ridx = board_of(j);
                mbar_wait_warp(&bar_c3[slot], (uint32_t)(j / NS) & 1u);
                PROF_T(5);
                tc_fence_after();
                const int y = m >> 3, x = m & 7;
                float v[8];
                tmem_ld_conv_sum(t_lane + slot * 128, v);
                if (y < 14 && x < 4) {
                    float o[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[e] = fmaxf(fmaf(v[e], K23, bias3[e]), 0.f);
                    uint4 c1, c2;
                    split8(o, c1, c2);
                    const int kc = (y * 4 + x) * 4 + cq;
                    *reinterpret_cast<uint4 *>(act3 + act3_off(0, n_tiles, ridx, kc)) = c1;
                    *reinterpret_cast<uint4 *>(act3 + act3_off(1, n_tiles, ridx, kc)) = c2;
                }
                tc_fence_before();
                PROF_T(6);
            }
        };
        auto phase_e1 = [&](int i) {
            // ---- E1(i): conv1 epilogue: bias + ReLU + split -> act1 (18x8 grid)
            if (i < n_local) {
                const int j = i, slot = j % NS;
                mbar_wait_warp(&bar_c1[slot], (uint32_t)(j / NS) & 1u);
                PROF_T(1);
                tc_fence_after();
                uint8_t *abase = smem + TCC_OFF_A1 + slot * TCC_ASLOT + cq * TCC_R * 16;
                const uint32_t t_c1 = t_lane + slot * 128;
                {
                    float w1[8], w2[8], o[8];
                    tmem_ld8x2(t_c1, w1, w2);
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[e] = fmaxf(fmaf(w2[e] + w1[e], K1, bias1[e]), 0.f);
                    uint4 c1, c2;
                    split8(o, c1, c2);
                    *reinterpret_cast<uint4 *>(abase + m * 16) = c1;
                    *reinterpret_cast<uint4 *>(abase + 4 * TCC_R * 16 + m * 16) = c2;
                }
                if (q == 0) {                                    // rows 128..143 sit in lanes 0..15 of the second M tile
                    float w1[8], w2[8], o[8];
                    tmem_ld8x2(t_c1 + 64, w1, w2);
                    if (lane < 16) {
#pragma unroll
                        for (int e = 0; e < 8; ++e) o[e] = fmaxf(fmaf(w2[e] + w1[e], K1, bias1[e]), 0.f);
                        uint4 c1, c2;
                        split8(o, c1, c2);
                        *reinterpret_cast<uint4 *>(abase + (128 + lane) * 16) = c1;
                        *reinterpret_cast<uint4 *>(abase + 4 * TCC_R * 16 + (128 + lane) * 16) = c2;
                    }
                }
                tc_fence_before();
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_a1[slot]);     // 32 same-address arrivals would serialise in the shared-memory pipe the MMAs read through
                PROF_T(2);
            }
        };
        for (int i = 0; i < n_iter; ++i) {
            phase_e2(i); phase_e3(i); phase_e1(i);
        }
        if (prof && do_prof) for (int i = 0; i < 16; ++i) if (i < 8 || i > 13) atomicAdd(&prof[i], (unsigned long long)pacc[i]);
    }
#undef PROF_T
    tc_fence_before();
    __syncthreads();
    if (warp == TCC_ISSUER) tmem_dealloc<TCC_TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------- fc pipeline
// [R, 16*KBLOCKS] x [16*KBLOCKS, N] over 128-row tiles, shared by k_tc_fc and k_tdc_fc.  Both operands are stored in HBM already in the
// canonical UMMA layout (A: the conv kernel's output, [split 2][tile][k chunk][row 128][8 fp16]; B: the packed fc1 weights), so one
// cp.async.bulk (1-D TMA) per operand block needs no tensor map.  Warp 0 streams the blocks into a STAGES-deep mbarrier ring, one lane
// of warp 1 issues three split MMAs per k block into N TMEM columns, warps 2-5 run the network's epilogue on the finished accumulator.
constexpr int FC_PIPE_THREADS = 192;
template <int N_, int KBLOCKS_, int STAGES_>
struct FcPipe {
    static constexpr int N = N_, KBLOCKS = KBLOCKS_, KCHUNKS = 2 * KBLOCKS, STAGES = STAGES_, TMEM_COLS = N;
    static constexpr int A_BYTES = 2 * 128 * 16;                 // one split of one k16 block of the A tile
    static constexpr int B_BYTES = 2 * N * 16;
    static constexpr int STAGE = 2 * A_BYTES + 2 * B_BYTES;
    static constexpr int OFF_BAR = STAGES * STAGE;
    static constexpr int OFF_EPI = OFF_BAR + 256;                 // the epilogue's constants
    static_assert((2 * STAGES + 2) * 8 + 4 <= 256, "barrier block overflows into the epilogue constants");
    static constexpr size_t ACT_TILE_BYTES = (size_t)2 * KCHUNKS * 2048;   // one 128-row tile of the A operand, both splits
};

// load_consts(t) copies the epilogue's constants to shared memory (thread t of FC_PIPE_THREADS).  epi(taddr, tile, row, n_req, drained) runs
// once per tile in every epilogue thread: taddr is the TMEM address of the thread's accumulator row, which holds request
// tile * 128 + row (>= n_req in the last tile's padding); it calls drained() once it has read the accumulator.
template <class P, class LoadConsts, class Epi>
__device__ __forceinline__ void fc_pipeline(const uint8_t *act, int n_tiles_alloc, const uint8_t *wfc, const int32_t *n_req_ptr,
                                            LoadConsts load_consts, Epi epi) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + P::OFF_BAR);   // [stage] operands landed
    uint64_t *empty = full + P::STAGES;                                  // [stage] operands consumed
    uint64_t *acc_full = empty + P::STAGES;                              // accumulator complete
    uint64_t *acc_empty = acc_full + 1;                                  // accumulator drained by the epilogue
    uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(acc_empty + 1);
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    __builtin_assume(t < FC_PIPE_THREADS);   // the kernels' launch bounds, which an inlined function does not see
    load_consts(t);
    if (t == 0) {
        for (int i = 0; i < P::STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, 128);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<P::TMEM_COLS>(tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const int n_req = *n_req_ptr;
    const int n_tiles = (n_req + 127) >> 7;
    if (warp == 0) {
        if (lane == 0) {   // ===== producer: bulk copies of the pre-laid-out operand blocks
            int stage = 0; uint32_t ph = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                for (int j = 0; j < P::KBLOCKS; ++j) {
                    mbar_wait(&empty[stage], ph ^ 1);
                    mbar_expect_tx(&full[stage], P::STAGE);
                    uint8_t *dst = smem + stage * P::STAGE;
#pragma unroll
                    for (int s = 0; s < 2; ++s) {
                        bulk_g2s(dst + s * P::A_BYTES, act + (((size_t)s * n_tiles_alloc + tile) * P::KCHUNKS + 2 * j) * 2048, P::A_BYTES, &full[stage]);
                        bulk_g2s(dst + 2 * P::A_BYTES + s * P::B_BYTES, wfc + ((size_t)s * P::KBLOCKS + j) * P::B_BYTES, P::B_BYTES, &full[stage]);
                    }
                    if (++stage == P::STAGES) { stage = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {   // ===== MMA issuer: D[128 x N] += A[128 x 16] * B[N x 16]^T, three split terms per k block
            const uint32_t idesc = umma_idesc_f16(128, P::N);
            int stage = 0; uint32_t ph = 0, aph = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                mbar_wait(acc_empty, aph ^ 1);
                tc_fence_after();
                uint32_t acc = 0;
                for (int j = 0; j < P::KBLOCKS; ++j) {
                    mbar_wait(&full[stage], ph);
                    tc_fence_after();
                    const uint32_t sbase = smem_u32(smem + stage * P::STAGE);
#pragma unroll
                    for (int term = 0; term < 3; ++term) {   // a1*b2, a2*b1, a1*b1 (small terms first)
                        const int sa = term == 1 ? 1 : 0, sb = term == 0 ? 1 : 0;
                        uint64_t ad = umma_desc(sbase + sa * P::A_BYTES, 128 * 16, 128);
                        uint64_t bd = umma_desc(sbase + 2 * P::A_BYTES + sb * P::B_BYTES, P::N * 16, 128);
                        umma_f16(tmem_base, ad, bd, idesc, acc);
                        acc = 1;
                    }
                    umma_commit(&empty[stage]);
                    if (++stage == P::STAGES) { stage = 0; ph ^= 1; }
                }
                umma_commit(acc_full);
                aph ^= 1;
            }
        }
    } else {   // ===== epilogue warps 2..5: TMEM quadrant = warp % 4, one row per thread
        const int q = warp & 3, row = q * 32 + lane;
        uint32_t aph = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            mbar_wait(acc_full, aph);
            tc_fence_after();
            epi(tmem_base + ((uint32_t)(q * 32) << 16), tile, row, n_req, [&] { tc_fence_before(); mbar_arrive(acc_empty); });
            aph ^= 1;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<P::TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------- fc kernel
using TcfPipe = FcPipe<256, ACT3_KCHUNKS / 2, 8>;
constexpr int TCF_SMEM = TcfPipe::OFF_EPI + (256 * 3 + 8) * 4;          // bias[256] | wout[2][256] | bout/ub/lb

__global__ void __launch_bounds__(FC_PIPE_THREADS, 1)
k_tc_fc(NetWeights W, TcWeights TW, const uint8_t *act3, int n_tiles_alloc, const uint2 *req, const int32_t *n_req_ptr, float2 *eval_out) {
    extern __shared__ __align__(128) uint8_t smem[];
    float *sBias = reinterpret_cast<float *>(smem + TcfPipe::OFF_EPI), *sWo = sBias + 256, *sTail = sWo + 512;
    auto load_consts = [&](int t) {
        for (int i = t; i < 256; i += FC_PIPE_THREADS) { sBias[i] = W.bfc1[i]; sWo[i] = W.wout[i]; sWo[256 + i] = W.wout[256 + i]; }
        if (t < 2) { sTail[t] = W.bout[t]; sTail[2 + t] = W.ub[t]; sTail[4 + t] = W.lb[t]; }
    };
    fc_pipeline<TcfPipe>(act3, n_tiles_alloc, TW.wfc, n_req_ptr, load_consts, [&](uint32_t taddr, int tile, int row, int n_req, auto drained) {
        float p0 = 0.f, p1 = 0.f;
#pragma unroll 1
        for (int c0 = 0; c0 < 256; c0 += 16) {
            float v[16];
            tmem_ld16(taddr + c0, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float h = fmaxf(v[j] * TC_UNSCALE + sBias[c0 + j], 0.f);   // model_vv.py:39-40
                p0 = fmaf(h, sWo[c0 + j], p0); p1 = fmaf(h, sWo[256 + c0 + j], p1);   // :41
            }
        }
        drained();
        const int ridx = tile * 128 + row;
        if (ridx < n_req) {
            float x0 = p0 + sTail[0], x1 = p1 + sTail[1];
            float s0 = 1.f / (1.f + expf(-x0)), s1 = 1.f / (1.f + expf(-x1));      // :42
            uint2 rq = req[ridx];
            eval_out[(size_t)rq.x * 8 + (rq.y >> 28)] =
                make_float2(__fadd_rn(__fmul_rn(s0, sTail[2]), sTail[4]), __fadd_rn(__fmul_rn(s1, sTail[3]), sTail[5]));   // :51
        }
    });
}

// ---------------------------------------------------------------------------------------------------- host side: weight packing
// Pure re-layout + fp16 splitting of the state_dict-order weights, shared by both tensor-core networks.
static inline void host_split2(float x, uint16_t *o) {   // x*scale = h1 + h2 in fp16
    __half h1 = __float2half_rn(x);
    __half h2 = __float2half_rn(x - __half2float(h1));
    memcpy(&o[0], &h1, 2); memcpy(&o[1], &h2, 2);
}
static inline float host_half_f(uint16_t h) { __half x; memcpy(&x, &h, 2); return __half2float(x); }

// conv1 (1 -> 32) as one K = 16 im2col MMA: [chunk 2][n = split*32 + cout][8], k = tap (9 or 16 taps; the rest zero)
static void pack_conv1(const float *cw, int taps, uint16_t *dst) {
    for (int c2 = 0; c2 < 2; ++c2)
        for (int n = 0; n < 32; ++n)
            for (int e = 0; e < 8; ++e) {
                const int tap = 8 * c2 + e;
                uint16_t s2[2] = {0, 0};
                if (tap < taps) host_split2(cw[n * taps + tap] * TC_SCALE_W, s2);
                for (int s = 0; s < 2; ++s) dst[((size_t)c2 * 64 + s * 32 + n) * 8 + e] = s2[s];
            }
}

// a taps x taps conv (32 -> 32) as a shift-GEMM: [(dy, half)][split][chunk][n = dx*32 + cout][8], N = taps * 32 (96 or 128)
static void pack_conv_shift(const float *cw, int taps, uint16_t *dst) {
    const int N = taps * 32;
    for (int dy = 0; dy < taps; ++dy)
        for (int hh = 0; hh < 2; ++hh)
            for (int c2 = 0; c2 < 2; ++c2)
                for (int dx = 0; dx < taps; ++dx)
                    for (int n = 0; n < 32; ++n)
                        for (int e = 0; e < 8; ++e) {
                            const int ci = 16 * hh + 8 * c2 + e;
                            uint16_t s2[2];
                            host_split2(cw[(n * 32 + ci) * taps * taps + dy * taps + dx] * TC_SCALE_W, s2);
                            for (int s = 0; s < 2; ++s)   // dy shifts the A operand and selects the block, dx is stacked along N
                                dst[(((((size_t)(dy * 2 + hh)) * 2 + s) * 2 + c2) * N + dx * 32 + n) * 8 + e] = s2[s];
                        }
}

// fc1 [N][K] with torch's flatten order k = c*pixels + p (32 channels, pixels = K / 32) as fc_pipeline's B operand:
// [split][k16 block][chunk][n][8], k' = pixel*32 + channel
static void pack_fc1(const float *fw, int N, int kblocks, uint16_t *dst) {
    const int K = kblocks * 16, pixels = K / 32;
    for (int j = 0; j < kblocks; ++j)
        for (int c2 = 0; c2 < 2; ++c2)
            for (int n = 0; n < N; ++n)
                for (int e = 0; e < 8; ++e) {
                    const int kp = j * 16 + c2 * 8 + e, p = kp >> 5, c = kp & 31;
                    uint16_t s2[2];
                    host_split2(fw[(size_t)n * K + c * pixels + p] * TC_SCALE_W, s2);
                    for (int s = 0; s < 2; ++s) dst[((((size_t)s * kblocks + j) * 2 + c2) * N + n) * 8 + e] = s2[s];
                }
}

constexpr size_t TC_PACKED_BYTES = TCC_W1BYTES + 2 * (size_t)TCC_WBYTES + (size_t)2 * TcfPipe::KBLOCKS * TcfPipe::B_BYTES;   // wc1 | wc2 | wc3 | wfc

// w = the state_dict-order weight vector of include/b200_tetris_mcts.h, packed into d_w (TC_PACKED_BYTES)
static int tc_prepare(const float *w, uint8_t *d_w, TcWeights &TW, cudaStream_t stream) {
    const float *c1w = w, *c2w = w + 288 + 32, *c3w = c2w + 9216 + 32, *f1w = c3w + 9216 + 32;
    std::vector<uint8_t> h(TC_PACKED_BYTES);
    TW.wc1 = d_w; TW.wc2 = d_w + TCC_W1BYTES; TW.wc3 = TW.wc2 + TCC_WBYTES; TW.wfc = TW.wc3 + TCC_WBYTES;
    auto at = [&](const uint8_t *d) { return reinterpret_cast<uint16_t *>(h.data() + (d - d_w)); };
    pack_conv1(c1w, 9, at(TW.wc1));
    pack_conv_shift(c2w, 3, at(TW.wc2));
    pack_conv_shift(c3w, 3, at(TW.wc3));
    pack_fc1(f1w, TcfPipe::N, TcfPipe::KBLOCKS, at(TW.wfc));
    if (cudaMemcpyAsync(d_w, h.data(), h.size(), cudaMemcpyHostToDevice, stream) != cudaSuccess) return 1;
    if (cudaStreamSynchronize(stream) != cudaSuccess) return 1;
    if (cudaFuncSetAttribute(k_tc_conv, cudaFuncAttributeMaxDynamicSharedMemorySize, TCC_SMEM) != cudaSuccess) return 1;
    if (cudaFuncSetAttribute(k_tc_fc, cudaFuncAttributeMaxDynamicSharedMemorySize, TCF_SMEM) != cudaSuccess) return 1;
    return 0;
}

}  // namespace b200
