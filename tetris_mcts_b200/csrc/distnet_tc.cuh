// distnet_tc.cuh — the reference's distributional value network (model/model_distributional.py:18-52) on Blackwell tensor cores, built from
// the pieces of valuenet_tc.cuh (same fp16 x 2 operand split, same scaling, same canonical no-swizzle K-major operand layouts):
//
//   k_tdc_conv  one persistent CTA per SM, four boards in flight.  The 20x10 observation gets the reference's two empty rows on top (22x10,
//               model_distributional.py:27).  conv1 4x4 (1->32): im2col [19x8 grid = 152 rows][16 taps] built by the front-end warp from the
//               observation key, ONE K=16 MMA per M tile (two tiles).  conv2 4x4 (32->32) as a shift-GEMM on the 8-wide grid: A = act1
//               started dy*8 rows later, the four horizontal taps stacked along N = 128, 4 dy x 2 channel halves x 3 split products = 24
//               tcgen05.mma (M=128, N=128, K=16); the epilogue sums the taps with three lane shuffles, applies bias + LeakyReLU(0.01),
//               re-splits and writes act2 (16x4 pixels x 32 channels = 2048 per board) to HBM in k_tdc_fc's tile layout.
//   k_tdc_fc    [R,2048] x [2048,128] on fc_pipeline (valuenet_tc.cuh) like k_tc_fc; epilogue: bias + LeakyReLU -> fc_v (128 x atoms, CUDA
//               cores, weights in shared memory) -> softmax (model_distributional.py:47-50) -> dist[game][atoms].
#pragma once
#include "valuenet_tc.cuh"
#include "distnet_simt.cuh"

namespace b200 {

constexpr int TDC_WORKERS = 512;                 // warps 0-15: the two epilogues
constexpr int TDC_ISSUER = TDC_WORKERS / 32;     // warp 16: MMA issuer (one elected lane)
constexpr int TDC_LOADER = TDC_ISSUER + 1;       // warp 17: observation keys -> conv1 operand
constexpr int TDC_THREADS = TDC_WORKERS + 64;
constexpr int TDC_R = 152;                       // act1 rows per board: the 19x8 grid (conv2 reads rows m + dy*8 <= 127 + 24)
constexpr int TDC_WBLOCK = 2 * 2 * 128 * 16;     // one (dy, channel half) block of conv2: [weight split 2][chunk 2][n = dx*32 + cout][16 B]
constexpr int TDC_WBYTES = 8 * TDC_WBLOCK;       // 65536
constexpr int TDC_W1BYTES = 2 * 64 * 16;         // conv1: [chunk 2][n = split*32 + cout][16 B], k = tap = dy*4 + dx
constexpr int TDC_SLOTS = 4;
constexpr int TDC_KEYS_AHEAD = 4;
constexpr int TDC_RUN = 4;
constexpr int TDC_ASLOT = 2 * 4 * TDC_R * 16;    // act1 of one board: [split][chunk 4][152 rows][16 B]
constexpr int TDC_IMROWS = 256;                  // two M = 128 tiles (152 rows used)
constexpr int TDC_IMSLOT = 2 * TDC_IMROWS * 16;
constexpr int TDC_OFF_W2 = 0;
constexpr int TDC_OFF_W1 = TDC_OFF_W2 + TDC_WBYTES;
constexpr int TDC_OFF_A1 = TDC_OFF_W1 + TDC_W1BYTES;
constexpr int TDC_OFF_IM = TDC_OFF_A1 + TDC_SLOTS * TDC_ASLOT;
constexpr int TDC_OFF_BIAS = TDC_OFF_IM + TDC_SLOTS * TDC_IMSLOT;    // 64 floats
constexpr int TDC_OFF_KEY = TDC_OFF_BIAS + 64 * 4;                   // TDC_SLOTS x 32 words: row table of the 22-row input (rows 0, 1 empty)
constexpr int TDC_OFF_BAR = TDC_OFF_KEY + TDC_SLOTS * 32 * 4;        // 4 x TDC_SLOTS mbarriers + tmem pointer
constexpr int TDC_SMEM = TDC_OFF_BAR + 4 * TDC_SLOTS * 8 + 16;
constexpr int TDC_TMEM_COLS = 512;               // 4 slots x 128 columns: conv1's two M tiles (2 x 64), then conv2's 128
constexpr int DACT2_KCHUNKS = 256;               // 2048 / 8
static_assert(TDC_SMEM <= 227 * 1024, "k_tdc_conv shared memory");

struct DnTcWeights {
    const uint8_t *wc1;   // TDC_W1BYTES
    const uint8_t *wc2;   // TDC_WBYTES, already in the shared-memory layout
    const uint8_t *wfc;   // [split 2][k16 block 128][chunk 2][n 128][16 B]
};

// act2 in HBM, FC-tile layout: [split][tile of 128 boards][k chunk 256][board 128][8 fp16], k' = (y*4 + x)*32 + c
__device__ __forceinline__ size_t dact2_off(int split, int n_tiles, int ridx, int kchunk) {
    return ((((size_t)split * n_tiles + (ridx >> 7)) * DACT2_KCHUNKS + kchunk) * 128 + (ridx & 127)) * 16;
}

// out[p] = D'[p][dx=0] + D'[p+1][dx=1] + D'[p+2][dx=2] + D'[p+3][dx=3] for the 8 couts of this warp's chunk
__device__ __forceinline__ void tmem_ld_conv4_sum(uint32_t taddr, float (&v)[8]) {
    float d0[8], d1[8], d2[8], d3[8];
    tmem_ld8x2(taddr, d0, d1);
    tmem_ld8x2(taddr + 64, d2, d3);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const float s1 = __shfl_down_sync(0xffffffffu, d1[e], 1), s2 = __shfl_down_sync(0xffffffffu, d2[e], 2), s3 = __shfl_down_sync(0xffffffffu, d3[e], 3);
        v[e] = ((s3 + s2) + s1) + d0[e];   // still scaled by 2^10 (see k_tc_conv: the scaling is folded into the bias fma)
    }
}

// conv2 = 24 tcgen05.mma of N = 128: for each (dy, channel half): a1*W1, a1*W2, a2*W1 into the same 128 columns
__device__ __forceinline__ void issue_dconv2(uint32_t tmem_d, uint32_t a_addr, uint32_t w_addr) {
    const uint64_t a0 = umma_desc(a_addr, TDC_R * 16, 128), b0 = umma_desc(w_addr, 128 * 16, 128);
    constexpr uint32_t idesc = umma_idesc_f16(128, 128);
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t a_hi = 2 * h * TDC_R + dy * 8, a_lo = a_hi + 4 * TDC_R;          // 16-byte units
            const uint32_t b_hi = (dy * 2 + h) * (TDC_WBLOCK / 16), b_lo = b_hi + 2 * 128;
            umma_f16(tmem_d, a0 + a_hi, b0 + b_hi, idesc, (dy | h) ? 1u : 0u);
            umma_f16(tmem_d, a0 + a_hi, b0 + b_lo, idesc, 1u);
            umma_f16(tmem_d, a0 + a_lo, b0 + b_hi, idesc, 1u);
        }
    }
}

__global__ void __launch_bounds__(TDC_THREADS, 1)
k_tdc_conv(DistNetWeights W, DnTcWeights TW, const uint2 *req, const int32_t *n_req_ptr, const uint32_t *keys, int M, uint8_t *act2, int n_tiles) {
    extern __shared__ __align__(128) uint8_t smem[];
    float *sB = reinterpret_cast<float *>(smem + TDC_OFF_BIAS);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + TDC_OFF_BAR);
    constexpr int NS = TDC_SLOTS;
    uint64_t *bar_c1 = bars, *bar_c2 = bars + NS;              // tensor core -> workers: layer of slot done
    uint64_t *bar_a0 = bars + 2 * NS, *bar_a1 = bars + 3 * NS;  // front end / workers -> issuer: operand of slot written
    uint32_t *sKey = reinterpret_cast<uint32_t *>(smem + TDC_OFF_KEY);
    uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(smem + TDC_OFF_BAR + 4 * NS * 8);
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    for (int i = t; i < TDC_WBYTES / 16; i += TDC_THREADS) reinterpret_cast<uint4 *>(smem + TDC_OFF_W2)[i] = reinterpret_cast<const uint4 *>(TW.wc2)[i];
    for (int i = t; i < TDC_W1BYTES / 16; i += TDC_THREADS) reinterpret_cast<uint4 *>(smem + TDC_OFF_W1)[i] = reinterpret_cast<const uint4 *>(TW.wc1)[i];
    for (int i = t; i < (TDC_OFF_BIAS - TDC_OFF_A1) / 16; i += TDC_THREADS) reinterpret_cast<uint4 *>(smem + TDC_OFF_A1)[i] = make_uint4(0, 0, 0, 0);
    if (t < 32) { sB[t] = W.b1[t]; sB[32 + t] = W.b2[t]; }
    if (t == 0) {
        for (int i = 0; i < 3 * NS; ++i) mbar_init(&bars[i], 1);                         // c1, c2 (tcgen05.commit), a0 (front-end warp)
        for (int i = 3 * NS; i < 4 * NS; ++i) mbar_init(&bars[i], TDC_WORKERS / 32);     // a1: one arrival per worker warp
        fence_barrier_init();
    }
    if (warp == TDC_ISSUER) tmem_alloc<TDC_TMEM_COLS>(tmem_ptr);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const int n_req = *n_req_ptr;
    // boards in runs of TDC_RUN consecutive requests per CTA (see k_tc_conv); board i of this CTA lives in slot i % 4:
    //   workers, iteration i :  E2(i-2) conv2 epilogue | E1(i) conv1 epilogue
    //   issuer,  iteration i :  [a1(i-1)] conv1(i) | conv2(i-1)      (conv1 first: its operand comes from the front-end warp, boards ahead)
    const int n_runs = (n_req + TDC_RUN - 1) / TDC_RUN;
    int n_local = 0;
    for (int run = blockIdx.x; run < n_runs; run += gridDim.x) n_local += min(TDC_RUN, n_req - run * TDC_RUN);
    auto board_of = [&](int i) -> int { return ((i / TDC_RUN) * (int)gridDim.x + (int)blockIdx.x) * TDC_RUN + (i % TDC_RUN); };
    if (warp == TDC_ISSUER) {
        if (lane == 0) {
            const uint32_t s_w1 = smem_u32(smem + TDC_OFF_W1), s_w2 = smem_u32(smem + TDC_OFF_W2);
            const uint32_t s_act = smem_u32(smem + TDC_OFF_A1), s_im = smem_u32(smem + TDC_OFF_IM);
            for (int i = 0; i < n_local + 1; ++i) {
                // a1(i-1): E1(i-1) done, and with it (program order of every worker warp) E2(i-3) — the last reader of the TMEM columns of
                // slot (i+1) % 4; conv1(i) writes slot i % 4, last read by E2(i-4)
                if (i >= 1) mbar_wait(&bar_a1[(i - 1) % NS], (uint32_t)((i - 1) / NS) & 1u);
                if (i < n_local) {                               // conv1 (model_distributional.py:20): im2col [256 x 16] x W1 [16 x 64], two M tiles
                    const int slot = i % NS;
                    mbar_wait(&bar_a0[slot], (uint32_t)(i / NS) & 1u);
                    tc_fence_after();
                    const uint64_t a0 = umma_desc(s_im + slot * TDC_IMSLOT, TDC_IMROWS * 16, 128), b0 = umma_desc(s_w1, 64 * 16, 128);
                    umma_f16(tmem_base + slot * 128, a0, b0, umma_idesc_f16(128, 64), 0u);
                    umma_f16(tmem_base + slot * 128 + 64, a0 + 128, b0, umma_idesc_f16(128, 64), 0u);
                    umma_commit(&bar_c1[slot]);
                }
                if (i >= 1) {                                    // conv2 (model_distributional.py:22): act1 on the 19x8 grid
                    const int j = i - 1, slot = j % NS;
                    tc_fence_after();
                    issue_dconv2(tmem_base + slot * 128, s_act + slot * TDC_ASLOT, s_w2);
                    umma_commit(&bar_c2[slot]);
                }
            }
        }
    } else if (warp == TDC_LOADER) {
        // front end: observation key (random 48-byte read) -> row table of the 22-row input -> im2col operand of conv1 (fp16, exact {-1,0,1}):
        // row p = y*8 + x of the 19x8 output grid, k = tap = dy*4 + dx; taps 0..7 in the first k chunk, 8..15 in the second
        uint2 rqs = make_uint2(0, 0);
        uint32_t kq[TDC_KEYS_AHEAD];
        auto fetch = [&](int i) -> uint32_t {
            if ((i & 31) == 0 && i + lane < n_local) rqs = req[board_of(i + lane)];
            const uint32_t gx = __shfl_sync(0xffffffffu, rqs.x, i & 31), gy = __shfl_sync(0xffffffffu, rqs.y, i & 31);
            return lane < 12 ? keys[((size_t)gx * M + (gy & 0x0fffffffu)) * KEY_WORDS + lane] : 0u;
        };
#pragma unroll
        for (int j = 0; j < TDC_KEYS_AHEAD; ++j) kq[j] = j < n_local ? fetch(j) : 0u;
        for (int i0 = 0; i0 < n_local; i0 += TDC_KEYS_AHEAD) {
#pragma unroll
            for (int j = 0; j < TDC_KEYS_AHEAD; ++j) {
                const int i = i0 + j;
                if (i >= n_local) break;
                const int slot = i % NS;
                // lane l < 22 holds input row l = board row l - 2 (rows 0, 1: the reference's padding): settled cells in bits 0..9, piece cells in 16..25
                const uint32_t kw = kq[j];
                const int br = lane - 2;
                const uint32_t rowpair = __shfl_sync(0xffffffffu, kw, (br >> 1) & 15), pcs = __shfl_sync(0xffffffffu, kw, 10);
                uint32_t tab = (rowpair >> ((br & 1) * 16)) & 0x3ffu;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t cell = (pcs >> (8 * k)) & 0xffu, pr = (cell * 205u) >> 11, pcol = cell - pr * 10u;
                    tab |= ((int)pr == br ? 1u : 0u) << (16 + pcol);
                }
                if (br < 0 || br >= 20) tab = 0u;
                if (i + TDC_KEYS_AHEAD < n_local) kq[j] = fetch(i + TDC_KEYS_AHEAD);
                if (i >= NS) mbar_wait_warp(&bar_c1[slot], (uint32_t)((i - NS) / NS) & 1u);     // conv1 of the slot's previous board has read its operand
                if (lane < 22) sKey[slot * 32 + lane] = tab;
                __syncwarp();
                uint8_t *im = smem + TDC_OFF_IM + slot * TDC_IMSLOT;
#pragma unroll
                for (int pp = 0; pp < 5; ++pp) {                 // 152 pixels over 32 lanes
                    const int p = pp * 32 + lane;
                    if (p < 152) {
                        const int y = p >> 3, x = p & 7;
                        uint32_t hv[16];
#pragma unroll
                        for (int dy = 0; dy < 4; ++dy) {
                            const uint32_t rw = sKey[slot * 32 + y + dy] >> x;
#pragma unroll
                            for (int dx = 0; dx < 4; ++dx)       // 1 settled, -1 falling piece, 0 empty; columns >= 10 (x = 7) read zero bits
                                hv[dy * 4 + dx] = ((rw >> dx) & 1u) * 0x3C00u | ((rw >> (16 + dx)) & 1u & (x + dx < 10 ? 1u : 0u)) * 0xBC00u;
                        }
                        *reinterpret_cast<uint4 *>(im + p * 16) =
                            make_uint4(hv[0] | (hv[1] << 16), hv[2] | (hv[3] << 16), hv[4] | (hv[5] << 16), hv[6] | (hv[7] << 16));
                        *reinterpret_cast<uint4 *>(im + TDC_IMROWS * 16 + p * 16) =
                            make_uint4(hv[8] | (hv[9] << 16), hv[10] | (hv[11] << 16), hv[12] | (hv[13] << 16), hv[14] | (hv[15] << 16));
                    }
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_a0[slot]);
            }
        }
    } else {
        // workers (512 threads): TMEM lane quadrant q, 8-cout chunk cq, pixel row m
        const int q = warp & 3, cq = warp >> 2, m = q * 32 + lane;
        const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + cq * 8;
        float bias1[8], bias2[8];                                  // pre-scaled by 16: leaky(x * 2^-10 + b) * 16 == leaky(fma(x, 2^-6, 16 b)) bit for bit
#pragma unroll
        for (int e = 0; e < 8; ++e) { bias1[e] = sB[cq * 8 + e] * TC_SCALE_A; bias2[e] = sB[32 + cq * 8 + e] * TC_SCALE_A; }
        constexpr float K2 = TC_UNSCALE * TC_SCALE_A, K1 = TC_SCALE_A / TC_SCALE_W;
        for (int i = 0; i < n_local + 2; ++i) {
            // ---- E2(i-2): conv2 epilogue: dx sum + bias + LeakyReLU + split -> act2 in HBM (FC tile layout)
            if (i >= 2) {
                const int j = i - 2, slot = j % NS, ridx = board_of(j);
                mbar_wait_warp(&bar_c2[slot], (uint32_t)(j / NS) & 1u);
                tc_fence_after();
                const int y = m >> 3, x = m & 7;
                float v[8];
                tmem_ld_conv4_sum(t_lane + slot * 128, v);
                if (x < 4) {
                    float o[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[e] = leaky(fmaf(v[e], K2, bias2[e]));
                    uint4 c1, c2;
                    split8(o, c1, c2);
                    const int kc = (y * 4 + x) * 4 + cq;
                    *reinterpret_cast<uint4 *>(act2 + dact2_off(0, n_tiles, ridx, kc)) = c1;
                    *reinterpret_cast<uint4 *>(act2 + dact2_off(1, n_tiles, ridx, kc)) = c2;
                }
                tc_fence_before();
            }
            // ---- E1(i): conv1 epilogue: bias + LeakyReLU + split -> act1 (19x8 grid)
            if (i < n_local) {
                const int slot = i % NS;
                mbar_wait_warp(&bar_c1[slot], (uint32_t)(i / NS) & 1u);
                tc_fence_after();
                uint8_t *abase = smem + TDC_OFF_A1 + slot * TDC_ASLOT + cq * TDC_R * 16;
                {
                    float w1[8], w2[8], o[8];
                    tmem_ld8x2(t_lane + slot * 128, w1, w2);
#pragma unroll
                    for (int e = 0; e < 8; ++e) o[e] = leaky(fmaf(w2[e] + w1[e], K1, bias1[e]));
                    uint4 c1, c2;
                    split8(o, c1, c2);
                    *reinterpret_cast<uint4 *>(abase + m * 16) = c1;
                    *reinterpret_cast<uint4 *>(abase + 4 * TDC_R * 16 + m * 16) = c2;
                }
                if (q == 0) {                                    // rows 128..151 sit in lanes 0..23 of the second M tile
                    float w1[8], w2[8], o[8];
                    tmem_ld8x2(t_lane + slot * 128 + 64, w1, w2);
                    if (lane < 24) {
#pragma unroll
                        for (int e = 0; e < 8; ++e) o[e] = leaky(fmaf(w2[e] + w1[e], K1, bias1[e]));
                        uint4 c1, c2;
                        split8(o, c1, c2);
                        *reinterpret_cast<uint4 *>(abase + (128 + lane) * 16) = c1;
                        *reinterpret_cast<uint4 *>(abase + 4 * TDC_R * 16 + (128 + lane) * 16) = c2;
                    }
                }
                tc_fence_before();
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_a1[slot]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == TDC_ISSUER) tmem_dealloc<TDC_TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------- fc1 + fc_v + softmax
using TdfPipe = FcPipe<128, DACT2_KCHUNKS / 2, 8>;
constexpr int TDF_ATOMS = 64;               // fc_v columns carried per thread (atoms <= 64, the rest zero)
constexpr int TDF_SMEM = TdfPipe::OFF_EPI + (128 + 128 * TDF_ATOMS + TDF_ATOMS) * 4;   // bias[128] | wv[128][64] | bv[64]

__global__ void __launch_bounds__(FC_PIPE_THREADS, 1)
k_tdc_fc(DistNetWeights W, DnTcWeights TW, const uint8_t *act2, int n_tiles_alloc, const uint2 *req, const int32_t *n_req_ptr, float *out) {
    extern __shared__ __align__(128) uint8_t smem[];
    float *sBias = reinterpret_cast<float *>(smem + TdfPipe::OFF_EPI), *sWv = sBias + 128, *sBv = sWv + 128 * TDF_ATOMS;
    const int atoms = W.atoms;
    auto load_consts = [=](int t) {   // by value: with `atoms` by reference the fc_v index below becomes a 64-bit multiply
        for (int i = t; i < 128; i += FC_PIPE_THREADS) sBias[i] = W.bf1[i];
        for (int i = t; i < 128 * TDF_ATOMS; i += FC_PIPE_THREADS) { const int k = i / TDF_ATOMS, a = i - k * TDF_ATOMS; sWv[i] = a < atoms ? W.wfv[(size_t)k * atoms + a] : 0.f; }
        if (t < TDF_ATOMS) sBv[t] = t < atoms ? W.bfv[t] : 0.f;
    };
    fc_pipeline<TdfPipe>(act2, n_tiles_alloc, TW.wfc, n_req_ptr, load_consts, [&](uint32_t taddr, int tile, int row, int n_req, auto drained) {
        float lg[TDF_ATOMS];
#pragma unroll
        for (int a = 0; a < TDF_ATOMS; ++a) lg[a] = sBv[a];
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 8) {
            float v[8];
            tmem_ld8(taddr + c0, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float h = leaky(v[j] * TC_UNSCALE + sBias[c0 + j]);          // model_distributional.py:43-44
                const float4 *wv = reinterpret_cast<const float4 *>(sWv + (c0 + j) * TDF_ATOMS);
#pragma unroll
                for (int a4 = 0; a4 < TDF_ATOMS / 4; ++a4) {                        // :45 (ascending k, like the CUDA-core kernel)
                    const float4 w4 = wv[a4];
                    lg[4 * a4] = fmaf(h, w4.x, lg[4 * a4]); lg[4 * a4 + 1] = fmaf(h, w4.y, lg[4 * a4 + 1]);
                    lg[4 * a4 + 2] = fmaf(h, w4.z, lg[4 * a4 + 2]); lg[4 * a4 + 3] = fmaf(h, w4.w, lg[4 * a4 + 3]);
                }
            }
        }
        drained();
        const int ridx = tile * 128 + row;
        if (ridx < n_req) {                                                        // F.softmax(x, 1), :47-50
            float mx = -INFINITY;
#pragma unroll
            for (int a = 0; a < TDF_ATOMS; ++a) if (a < atoms) mx = fmaxf(mx, lg[a]);
            float sum = 0.f;
#pragma unroll
            for (int a = 0; a < TDF_ATOMS; ++a) if (a < atoms) { lg[a] = expf(lg[a] - mx); sum += lg[a]; }
            float *dst = out + (size_t)req[ridx].x * atoms;
#pragma unroll
            for (int a = 0; a < TDF_ATOMS; ++a) if (a < atoms) dst[a] = lg[a] / sum;
        }
    });
}

// ---------------------------------------------------------------------------------------------------- host side
constexpr size_t DN_TC_PACKED_BYTES = TDC_W1BYTES + (size_t)TDC_WBYTES + (size_t)2 * TdfPipe::KBLOCKS * TdfPipe::B_BYTES;   // wc1 | wc2 | wfc

// w = the state_dict-order weight vector of model_distributional.py (see dn_relayout), packed into d_w (DN_TC_PACKED_BYTES)
static int dn_tc_prepare(const float *w, uint8_t *d_w, DnTcWeights &TW, cudaStream_t stream) {
    const float *c1w = w, *c2w = c1w + 512 + 32, *f1w = c2w + 16384 + 32;
    std::vector<uint8_t> h(DN_TC_PACKED_BYTES);
    TW.wc1 = d_w; TW.wc2 = d_w + TDC_W1BYTES; TW.wfc = TW.wc2 + TDC_WBYTES;
    auto at = [&](const uint8_t *d) { return reinterpret_cast<uint16_t *>(h.data() + (d - d_w)); };
    pack_conv1(c1w, 16, at(TW.wc1));
    pack_conv_shift(c2w, 4, at(TW.wc2));
    pack_fc1(f1w, TdfPipe::N, TdfPipe::KBLOCKS, at(TW.wfc));
    if (cudaMemcpyAsync(d_w, h.data(), h.size(), cudaMemcpyHostToDevice, stream) != cudaSuccess) return 1;
    if (cudaStreamSynchronize(stream) != cudaSuccess) return 1;
    if (cudaFuncSetAttribute(k_tdc_conv, cudaFuncAttributeMaxDynamicSharedMemorySize, TDC_SMEM) != cudaSuccess) return 1;
    if (cudaFuncSetAttribute(k_tdc_fc, cudaFuncAttributeMaxDynamicSharedMemorySize, TDF_SMEM) != cudaSuccess) return 1;
    return 0;
}

}  // namespace b200
