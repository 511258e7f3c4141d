// tcgen05 tensor-core path of the ConvBlock and of the plain (1x1 / k-tap) weight-normed convolutions: forward,
// data-gradient and weight-gradient as implicit GEMMs with fp32-equivalent accuracy from split-bf16 operands.
// Every fp32 operand is split into bf16 planes p0 = bf16(x), p1 = bf16(x - p0) and each K-step issues
// p0*p0 + p0*p1 + p1*p0 (operand error ~2^-17; single-pass TF32 would miss the rtol=1e-3/atol=1e-4 parity bar after
// ~30 blocks).  The tensor core adds each MMA into the fp32 accumulator with truncation (bias ~N_mma x 2^-25), so the
// main term p0*p0 and the 2^-8-smaller cross terms accumulate in two separate TMEM accumulators that the epilogue
// adds in fp32 (tools/precision_report.py).
//
//   GATED : D[t, (a|b) c] = sum_{j,ci} Xd[b, t+off_j, ci] * W[j, (a|b) c, ci]    M = 128 time steps, N = 64 a | 64 b
//   CONV  : D[t, n]       = sum_{j,kc} A[b, t+off_j, kc]  * W[j, n, kc]           M = 128 time steps, N = 64 or 128
//           (plain conv forward with bias/ReLU, and every data gradient: A = dY or dAB, W = transposed weight)
//   WGRAD : D[m, n] (j)   = sum_{b,t}  dY[b, t, m] * Xd[b, t+off_j, n]            MN-major operands, M = 128, N <= 256
//
// Operands are bf16 (B,T,C) planes fetched by TMA as K-major tiles of 128 rows x BK (BK = 64: 128-byte rows,
// SWIZZLE_128B -- wherever the channel count is a multiple of 64; BK = 32: 64-byte rows, SWIZZLE_64B); the conv's zero
// padding, the causal shift, ragged T / channel tails are TMA out-of-bounds zero fill.  The hi and lo weight planes sit
// back to back in a stage, so p0(A) x [p0(W) ; p1(W)] is ONE N = 2*NCOLS MMA filling the main | cross accumulators,
// followed by p1(A) x p0(W) into the cross accumulator.
//
// tc_conv_kernel is PERSISTENT: one CTA per SM walks a static round-robin list of output tiles; TMEM holds two
// accumulator sets, so the epilogue warps drain tile n while the MMA thread accumulates tile n+1 and the TMA ring
// streams across tile boundaries.  Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer,
// warps 2-5 = epilogue (TMEM -> registers -> fused math -> stores coalesced along T).
#include "tc_common.cuh"
#include "../../include/dv3b200.h"

namespace dv3 {

using namespace tc;

constexpr int TC_THREADS = 192;
constexpr int MAX_TAPS_TC = 8;
constexpr int SMEM_LIMIT = 232448;          // 227 KB opt-in dynamic shared memory per CTA

enum { TC_GATED = 0, TC_CONV = 1 };

struct TcMaps { CUtensorMap a[2]; CUtensorMap b[2]; };

struct TcParams {
    int T, B;
    int Kc;                    // contraction channels per tap
    int Nc;                    // output channels (GATED: C per half)
    int rows_per_tap;          // rows of the weight matrix per tap (GATED: 2C, CONV: Nc)
    int k, kb_n;               // taps; K blocks per tap
    int tap_off[MAX_TAPS_TC];
    // gated epilogue
    const float* bias; const float* spk; const float* res;
    float* y; float* save_a; float* save_s;
    int gate_mode, residual;
    // conv epilogue: out = acc*dropmask + bias + addend ; relu
    float* out; const float* e1; const float* e2; float alpha; int addmode, relu;
    float p_drop; const unsigned long long* seed_ptr; uint32_t salt;
    // Compensation of the tensor core's truncating accumulation: every tcgen05.mma adds its K = 16 partial product
    // into the fp32 accumulator rounding TOWARD ZERO, an expected relative loss of ~0.35 * 2^-23 per event on the
    // running sum; over the n_mma events of one output that is a systematic shrink of ~gcoef * n_mma (measured,
    // tools/precision_presets.py).  The epilogue multiplies the main accumulator by gmain = 1 + gcoef * n_mma (the
    // cross-term accumulator is 2^-8 smaller: its loss is below fp32 resolution).
    float gmain;
    uint32_t idesc_fmt;        // a_format / b_format bits of the instruction descriptor (fp16 forward, bf16 gradients)
};

template <int BK> struct SwizzleOf;
template <> struct SwizzleOf<64> { static constexpr uint32_t layout = 2, sbo = 1024; };   // SWIZZLE_128B
template <> struct SwizzleOf<32> { static constexpr uint32_t layout = 4, sbo = 512; };    // SWIZZLE_64B

template <int BK>
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);                 // start address / 16
    d |= (uint64_t)(SwizzleOf<BK>::sbo >> 4) << 32;          // stride between 8-row swizzle atoms
    d |= (uint64_t)1 << 46;                                  // sm_100 descriptor version
    d |= (uint64_t)SwizzleOf<BK>::layout << 61;
    return d;
}

// BR = rows of one B-operand box (128, or 64 for problems too small to fill the machine with 128-wide tiles)
template <int NBOX, int BK, int BR>
struct TcCfg {
    static constexpr int TILE = 128 * BK * 2;            // A tile (128 rows)
    static constexpr int TILE_B = BR * BK * 2;           // one B box
    static constexpr int STAGE = 2 * (TILE + NBOX * TILE_B);
    static constexpr int STAGES_RAW = (SMEM_LIMIT - 2048) / STAGE;
    static constexpr int STAGES = STAGES_RAW > 6 ? 6 : STAGES_RAW;
    static constexpr int SMEM = STAGES * STAGE + 1024 + 512;   // + alignment slack + barriers
    static constexpr int NCOLS = BR * NBOX;              // columns per accumulator; (main, cross) x two sets
};
// Ring depths of the instantiations the host code launches (<NBOX, BK, BR>), pinned so a change is deliberate.
static_assert(TcCfg<2, 64, 64>::STAGES == 3, "gated <0,2,64,64>");
static_assert(TcCfg<1, 64, 128>::STAGES == 3, "conv <1,1,128,64>");
static_assert(TcCfg<1, 64, 64>::STAGES == 4, "conv <1,1,64,64>");
static_assert(TcCfg<1, 32, 128>::STAGES == 6, "conv <1,1,128,32>");
static_assert(TcCfg<1, 32, 64>::STAGES == 6, "conv <1,1,64,32>");

// main + cross accumulator -> registers, summed in fp32 (round-to-nearest)
// gmain = 1 + (expected relative truncation loss of the main accumulator), see TcParams::gmain
__device__ __forceinline__ void tmem_ld_add(uint32_t taddr, int cross_off, float* v, float gmain) {
    float c[32];
    tmem_ld_32x32(taddr, v);
    tmem_ld_32x32(taddr + cross_off, c);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = fmaf(c[i], LO_INV, v[i] * gmain);       // lo planes carry a 2^11 scale
}

// ---- epilogues -----------------------------------------------------------------------------------------------
// NOTE on the epilogue loads: residual / addend / bias reads go through __ldg (ld.global.nc) and are issued as a
// batch of 32 independent loads BEFORE the dependent math and stores of the chunk.  With plain loads the compiler
// must order every load after the previous iteration's stores (possible aliasing), which serialised 128
// global-memory round trips per thread (ncu: 40 % of the stall samples sat on the first use of these loads).
template <int BR, int NCOLS>
__device__ __forceinline__ void epilogue_gated(const TcParams& p, uint32_t taddr, int a_row0, int a_z, int b_row0,
                                               int row) {
    const int t = a_row0 + row, b = a_z, C = p.Nc;
    const bool tv = t < p.T;
    const float* __restrict__ bias = p.bias;
    const float* __restrict__ res = p.res;
    const float* __restrict__ spk = p.spk;
    float* __restrict__ yo = p.y;
    float* __restrict__ ao = p.save_a;
    float* __restrict__ so = p.save_s;
    const bool need_res = (p.gate_mode != 0) || p.residual;
    const size_t base = ((size_t)b * C + b_row0) * p.T + (tv ? t : 0);
    for (int c32 = 0; c32 < BR; c32 += 32) {
        float va[32], vb[32], rr[32];
        tmem_ld_add(taddr + c32, NCOLS, va, p.gmain);
        tmem_ld_add(taddr + BR + c32, NCOLS, vb, p.gmain);
        if (tv) {
            const size_t cb = base + (size_t)c32 * p.T;
#pragma unroll
            for (int i = 0; i < 32; ++i) rr[i] = need_res ? __ldg(&res[cb + (size_t)i * p.T]) : 0.f;
            if (spk) {
#pragma unroll
                for (int i = 0; i < 32; ++i) va[i] += __ldg(&spk[cb + (size_t)i * p.T]);
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int c = b_row0 + c32 + i;
                const size_t idx = cb + (size_t)i * p.T;
                const float a = va[i] + __ldg(&bias[c]);
                const float s = sigmoidf_(vb[i] + __ldg(&bias[C + c]));
                float y;
                if (p.gate_mode == 0) {
                    y = a * s;
                    if (p.residual) y = (y + rr[i]) * 0.70710678118654752f;
                } else {
                    y = s * a + (1.f - s) * rr[i];
                }
                yo[idx] = y;
                if (ao) ao[idx] = a;
                if (so) so[idx] = s;
            }
        }
    }
}

template <int NCOLS>
__device__ __forceinline__ void epilogue_conv(const TcParams& p, uint32_t taddr, int a_row0, int a_z, int b_row0,
                                              int row) {
    const int t = a_row0 + row, b = a_z;
    const bool tv = t < p.T;
    const DropCfg drop = make_drop(p.p_drop, p.seed_ptr, p.salt);
    const float* __restrict__ bias = p.bias;
    const float* __restrict__ e1 = p.e1;
    const float* __restrict__ e2 = p.e2;
    float* __restrict__ out = p.out;
    for (int c32 = 0; c32 < NCOLS; c32 += 32) {
        float v[32], x1[32], x2[32];
        tmem_ld_add(taddr + c32, NCOLS, v, p.gmain);
        const int n0 = b_row0 + c32;
        const size_t cb = ((size_t)b * p.Nc + n0) * p.T + (tv ? t : 0);
        if (tv) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const bool ok = n0 + i < p.Nc;
                x1[i] = (p.addmode != 0 && ok) ? __ldg(&e1[cb + (size_t)i * p.T]) : 0.f;
                x2[i] = (p.addmode == 2 && ok) ? __ldg(&e2[cb + (size_t)i * p.T]) : 0.f;
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int n = n0 + i;
                if (n < p.Nc) {
                    const size_t idx = cb + (size_t)i * p.T;
                    float g = v[i] * drop_scale(drop, (uint32_t)idx);
                    if (bias) g += __ldg(&bias[n]);
                    if (p.addmode == 1) g += p.alpha * x1[i];
                    else if (p.addmode == 2) g += x1[i] * (1.f - x2[i]);
                    if (p.relu) g = fmaxf(g, 0.f);
                    out[idx] = g;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// GATED / CONV kernel (persistent, see file header).  N per tile is limited to 128 columns (4 x 128 = 512 TMEM columns).
// ------------------------------------------------------------------------------------------------
template <int MODE, int NBOX, int BR, int BK>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_conv_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcParams p, int tiles_x, int tiles_y,
               int num_tiles) {
    pdl_trigger();
    using Cfg = TcCfg<NBOX, BK, BR>;
    constexpr int TILE = Cfg::TILE, TILE_B = Cfg::TILE_B, STAGE = Cfg::STAGE, STAGES = Cfg::STAGES, NCOLS = Cfg::NCOLS;
    constexpr int B_OFF = 2 * TILE;
    static_assert(4 * NCOLS <= 512, "two accumulator sets of (main + cross) must fit in TMEM");
    static_assert(STAGES >= 2, "pipeline needs at least two stages");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE);
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;          // [2] accumulator set ready for the epilogue
    uint64_t* tempty = tfull + 2;              // [2] accumulator set drained
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tempty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_iters = p.k * p.kb_n;

    if (threadIdx.x == 0) {
        prefetch_tmap(&maps.a[0]); prefetch_tmap(&maps.a[1]); prefetch_tmap(&maps.b[0]); prefetch_tmap(&maps.b[1]);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 128); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<4 * NCOLS>(tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    pdl_wait();                    // everything above overlapped the previous kernel's tail; global memory from here

    // tile id -> (time tile, channel tile, batch); channel tiles vary fastest so that concurrently running CTAs share
    // the activation tile in L2
    auto decode = [&](int tile, int& a_row0, int& a_z, int& b_row0, int& b_row1) {
        const int ty = tile % tiles_y, r = tile / tiles_y;
        const int tx = r % tiles_x;
        a_z = r / tiles_x;
        a_row0 = tx * 128;
        if (MODE == TC_GATED) { b_row0 = ty * BR; b_row1 = p.Nc + ty * BR; }
        else { b_row0 = ty * BR * NBOX; b_row1 = b_row0 + BR; }
    };

    if (warp == 0 && lane == 0) {
        int it = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            int a_row0, a_z, b_row0, b_row1;
            decode(tile, a_row0, a_z, b_row0, b_row1);
            for (int kit = 0; kit < n_iters; ++kit, ++it) {
                const int s = it % STAGES, ph = (it / STAGES) & 1;
                mbar_wait(&empty[s], ph ^ 1);
                uint8_t* st = smem + s * STAGE;
                const int j = kit / p.kb_n, kb = kit - j * p.kb_n;
                const int ax = kb * BK, ay = a_row0 + p.tap_off[j];
                const int by0 = j * p.rows_per_tap + b_row0, by1 = j * p.rows_per_tap + b_row1;
                mbar_arrive_expect_tx(&full[s], STAGE);
#pragma unroll
                for (int pl = 0; pl < 2; ++pl) {
                    tma_load_3d(st + pl * TILE, &maps.a[pl], &full[s], ax, ay, a_z);
                    uint8_t* bdst = st + B_OFF + pl * NBOX * TILE_B;
                    tma_load_3d(bdst, &maps.b[pl], &full[s], ax, by0, 0);
                    if (NBOX == 2) tma_load_3d(bdst + TILE_B, &maps.b[pl], &full[s], ax, by1, 0);
                }
            }
        }
    } else if (warp == 1 && lane == 0) {
        const uint32_t idesc = make_idesc_mn(128, NCOLS) | p.idesc_fmt, idesc2 = make_idesc_mn(128, 2 * NCOLS) | p.idesc_fmt;
        int it = 0, tcount = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++tcount) {
            const int a = tcount & 1, aph = (tcount >> 1) & 1;
            mbar_wait(&tempty[a], aph ^ 1);                         // the epilogue has drained this accumulator set
            tc_fence_after();
            const uint32_t acc = tmem_base + a * 2 * NCOLS;
            for (int kit = 0; kit < n_iters; ++kit, ++it) {
                const int s = it % STAGES, ph = (it / STAGES) & 1;
                mbar_wait(&full[s], ph);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + s * STAGE);
                const uint64_t da0 = make_desc<BK>(sa), da1 = make_desc<BK>(sa + TILE);
                const uint64_t db0 = make_desc<BK>(sa + B_OFF);         // plane 1 follows plane 0: rows [NCOLS, 2 NCOLS)
#pragma unroll
                for (int kk = 0; kk < BK / 16; ++kk) {
                    const uint64_t adv = (uint64_t)(kk * 2);
                    umma_bf16(acc, da0 + adv, db0 + adv, idesc2, (kit | kk) != 0);     // p0 x [p0 ; p1] -> main | cross
                    umma_bf16(acc + NCOLS, da1 + adv, db0 + adv, idesc, 1);
                }
                umma_commit(&empty[s]);
            }
            umma_commit(&tfull[a]);
        }
    } else if (warp >= 2) {
        const int q = warp & 3, row = q * 32 + lane;
        int tcount = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++tcount) {
            int a_row0, a_z, b_row0, b_row1;
            decode(tile, a_row0, a_z, b_row0, b_row1);
            const int a = tcount & 1, aph = (tcount >> 1) & 1;
            mbar_wait(&tfull[a], aph);
            tc_fence_after();
            const uint32_t taddr = tmem_base + a * 2 * NCOLS + ((uint32_t)(q * 32) << 16);
            if (MODE == TC_GATED) epilogue_gated<BR, NCOLS>(p, taddr, a_row0, a_z, b_row0, row);
            else epilogue_conv<NCOLS>(p, taddr, a_row0, a_z, b_row0, row);
            tc_fence_before();
            mbar_arrive(&tempty[a]);                                // 128 arrivals release the set to the MMA thread
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<4 * NCOLS>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// Weight gradient straight from the (B,T,C) planes the forward / data-gradient GEMMs already use:
//     D[m, n] (tap j) = sum_{b,t} dY[b, t, m] * Xd[b, t + off_j, n]
// Both operands are "MN-major" here (channels contiguous, the contraction index t is the row): 64-channel x 32-row
// TMA boxes (128-byte rows, SWIZZLE_128B), UMMA descriptors with the MN-major canonical layout
// ((64 channels contiguous, chunk stride LBO), (8 rows x 128 B, group stride SBO)) and a_major = b_major = 1 in the
// instruction descriptor.  The tap shift is a ROW coordinate of the TMA box (any alignment, out-of-bounds rows are
// zero = the conv padding), so no time-shifted copies of the input are needed.
// ------------------------------------------------------------------------------------------------
struct TcMnParams {
    int T, B, Mw, Nw, k;
    int tap_off[MAX_TAPS_TC];
    int nsplit, batches_per_split, kb_n;      // kb_n = 32-row time chunks per utterance
    float* dw; long long split_stride;
    int msplit; long long s_m, s_mh, s_n, s_j;
    float gcoef;                              // see TcParams::gmain (n_mma = 2 per 32-row time chunk)
};

__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
    return d;
}

template <int NBOX>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_wgrad_mn_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcMnParams p) {
    pdl_trigger();
    constexpr int BOX = 64 * 32 * 2;                     // 64 channels x 32 time steps of bf16 = 4 KB
    constexpr int A_PL = 2 * BOX, B_PL = 2 * NBOX * BOX; // per plane: 128 rows of M, 128*NBOX columns of N
    constexpr int STAGE = 2 * (A_PL + B_PL);
    constexpr int STAGES = ((SMEM_LIMIT - 2048) / STAGE) > 6 ? 6 : ((SMEM_LIMIT - 2048) / STAGE);
    constexpr int NCOLS = 128 * NBOX;
    constexpr uint32_t LBO = 4096, SBO = 1024;           // 64-channel chunks one TMA box apart; 8-row groups 1 KB apart
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE);
    uint64_t* empty = full + STAGES;
    uint64_t* tmem_full = empty + STAGES;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_full + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    const int wg_j = blockIdx.z % p.k, wg_split = blockIdx.z / p.k;
    const int m0 = blockIdx.y * 128, n0 = blockIdx.x * 128 * NBOX;
    const int b_beg = wg_split * p.batches_per_split;
    int b_end = b_beg + p.batches_per_split; if (b_end > p.B) b_end = p.B;
    const int n_iters = (b_end > b_beg ? b_end - b_beg : 0) * p.kb_n;

    if (threadIdx.x == 0) {
        prefetch_tmap(&maps.a[0]); prefetch_tmap(&maps.a[1]); prefetch_tmap(&maps.b[0]); prefetch_tmap(&maps.b[1]);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tmem_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<2 * NCOLS>(tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    pdl_wait();

    if (warp == 0 && lane == 0) {
        for (int it = 0; it < n_iters; ++it) {
            const int s = it % STAGES, ph = (it / STAGES) & 1;
            mbar_wait(&empty[s], ph ^ 1);
            uint8_t* st = smem + s * STAGE;
            const int bi = it / p.kb_n, tc_ = it - bi * p.kb_n;
            const int b = b_beg + bi, t0 = tc_ * 32;
            mbar_arrive_expect_tx(&full[s], STAGE);
#pragma unroll
            for (int pl = 0; pl < 2; ++pl) {
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    tma_load_3d(st + pl * A_PL + h * BOX, &maps.a[pl], &full[s], m0 + h * 64, t0, b);
#pragma unroll
                for (int q = 0; q < 2 * NBOX; ++q)
                    tma_load_3d(st + 2 * A_PL + pl * B_PL + q * BOX, &maps.b[pl], &full[s], n0 + q * 64,
                                t0 + p.tap_off[wg_j], b);
            }
        }
    } else if (warp == 1 && lane == 0) {
        // A = gradient planes, B = the bf16 copy of the forward operand planes; both MN-major
        constexpr uint32_t idesc = make_idesc_bf16(128, NCOLS) | (1u << 15) | (1u << 16);
        for (int it = 0; it < n_iters; ++it) {
            const int s = it % STAGES, ph = (it / STAGES) & 1;
            mbar_wait(&full[s], ph);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + s * STAGE);
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {                        // 2 x UMMA_K(16 rows of 128 B)
                const uint32_t ko = kk * 16 * 128;
                const uint64_t a0 = make_desc_mn(sa + ko, LBO, SBO);
                const uint64_t a1 = make_desc_mn(sa + A_PL + ko, LBO, SBO);
                const uint64_t b0 = make_desc_mn(sa + 2 * A_PL + ko, LBO, SBO);
                const uint64_t b1 = make_desc_mn(sa + 2 * A_PL + B_PL + ko, LBO, SBO);
                umma_bf16(tmem_base, a0, b0, idesc, (it | kk) != 0);
                umma_bf16(tmem_base + NCOLS, a0, b1, idesc, (it | kk) != 0);
                umma_bf16(tmem_base + NCOLS, a1, b0, idesc, 1);
            }
            umma_commit(&empty[s]);
        }
        umma_commit(tmem_full);
    } else if (warp >= 2) {
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        const int q = warp & 3, row = q * 32 + lane;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
        const int m = m0 + row;
        float* __restrict__ out = p.dw + (size_t)wg_split * p.split_stride + (size_t)wg_j * p.s_j;
        const size_t ma = (size_t)(m % p.msplit) * p.s_m + (size_t)(m / p.msplit) * p.s_mh;
        // partials with unit stride along n ([split][j][m][n]): each thread owns a contiguous run -> float4 stores
        const bool vec = (p.s_n == 1) && ((p.Nw & 3) == 0) &&
                         (((ma + (size_t)wg_j * p.s_j + (size_t)wg_split * p.split_stride) & 3) == 0);
        for (int c32 = 0; c32 < NCOLS; c32 += 32) {
            float v[32];
            tmem_ld_add(taddr + c32, NCOLS, v, 1.f + p.gcoef * (float)(2 * n_iters));
            if (m >= p.Mw) continue;
            const int nn = n0 + c32;
            if (n_iters == 0) {
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = 0.f;
            }
            if (vec && nn + 32 <= p.Nw) {
#pragma unroll
                for (int i = 0; i < 32; i += 4)
                    *reinterpret_cast<float4*>(&out[ma + nn + i]) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
            } else {
#pragma unroll
                for (int i = 0; i < 32; ++i)
                    if (nn + i < p.Nw) out[ma + (size_t)(nn + i) * p.s_n] = v[i];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<2 * NCOLS>(tmem_base);
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static const EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres);
        return (e == cudaSuccess) ? (EncodeTiledFn)f : (EncodeTiledFn) nullptr;
    }();
    return fn;
}

// bf16 3-D tensor map; box = (box0, box1, 1); swizzle chosen from the box width (64 or 128 bytes)
int encode_tmap_bf16_3d(CUtensorMap* map, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                        uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0, uint32_t box1) {
    const EncodeTiledFn enc = encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return 1; }
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
    cuuint32_t box[3] = {box0, box1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapSwizzle sw = box0 * 2 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): dims=(%llu,%llu,%llu) strides=(%llu,%llu) box=(%u,%u)", (int)r,
                  (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
                  (unsigned long long)stride1_bytes, (unsigned long long)stride2_bytes, box0, box1);
        return 1;
    }
    return 0;
}

template <typename K>
static int ensure_smem(K kern, int bytes, const char* what) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) { set_error("%s: cannot set %d B dynamic smem: %s", what, bytes, cudaGetErrorString(e)); return 1; }
    return 0;
}

template <int MODE, int NBOX, int BR, int BK>
static int launch_conv(const TcMaps& maps, const TcParams& p, int tiles_x, int tiles_y, int batch, cudaStream_t st,
                       const char* what) {
    using Cfg = TcCfg<NBOX, BK, BR>;
    auto kern = tc_conv_kernel<MODE, NBOX, BR, BK>;
    static const int configured = ensure_smem(kern, Cfg::SMEM, what);       // once per instantiation, thread-safe
    if (configured) return 1;
    const int sms = config().sms;
    const int num_tiles = tiles_x * tiles_y * batch;
    const int grid = num_tiles < sms ? num_tiles : sms;
    cudaError_t e = launch_k(kern, dim3(grid), dim3(TC_THREADS), (size_t)Cfg::SMEM, st, maps, p, tiles_x, tiles_y,
                             num_tiles);
    if (e != cudaSuccess) { set_error("%s: launch failed: %s", what, cudaGetErrorString(e)); return 1; }
    return check_launch(what);
}

static void fill_taps_tc(int* tap_off, int k, int dilation, int causal, bool transpose) {
    const int padl = causal ? (k - 1) * dilation : (k - 1) / 2 * dilation;
    for (int j = 0; j < MAX_TAPS_TC; ++j)
        tap_off[j] = j < k ? (transpose ? (padl - j * dilation) : (j * dilation - padl)) : 0;
}

// plane p of a [nplanes][...] bf16 buffer
static inline const void* plane(const void* base, int pl, long long plane_elems) {
    return (const char*)base + (size_t)pl * plane_elems * 2;
}

}  // namespace dv3

using namespace dv3;

extern "C" {

// 1 if the tensor-core ConvBlock path supports this block shape (else the caller uses the exact-fp32 kernels)
int dv3_tc_supported(int B, int C, int T, int k) {
    return (C % 128 == 0) && T >= 1 && k >= 1 && k <= MAX_TAPS_TC && B >= 1 && B <= 65535;
}
// plain convs: any channel counts (planes are padded to a multiple of 8 channels); k-tap convs need
// Cout % 128 == 0 so a weight box never straddles two taps
int dv3_tc_conv_supported(int B, int Cin, int Cout, int T, int k) {
    return T >= 1 && k >= 1 && k <= MAX_TAPS_TC && B >= 1 && B <= 65535 && (k == 1 || Cout % 128 == 0) && Cin >= 8 &&
           Cout >= 1;
}

// Gated forward.  xd: [2][B][T][C] bf16 planes of the (dropped-out) input; w: [2][k][2C][C] bf16 planes of the
// normalised weight; the rest as dv3_convblock_fwd.  64-channel tiles (64 a | 64 b columns), BK = 64.
int dv3_tc_convblock_fwd(const void* xd, const void* w, int npl, const float* bias, const float* spk,
                         const float* res, float* y, float* save_a, float* save_s, int B, int C, int T, int k,
                         int dilation, int causal, int mode, int residual, const void* reserved, void* stream) {
    DV3_REQUIRE(reserved == nullptr, "tc_convblock_fwd: reserved must be NULL");
    DV3_REQUIRE(dv3_tc_supported(B, C, T, k), "tc_convblock_fwd: unsupported shape B=%d C=%d T=%d k=%d", B, C, T, k);
    DV3_REQUIRE(npl == 2, "tc_convblock_fwd: npl must be 2");
    TcMaps maps;
    const int t_tiles = (T + 127) / 128;
    for (int pl = 0; pl < 2; ++pl) {
        if (encode_tmap_bf16_3d(&maps.a[pl], plane(xd, pl, (long long)B * T * C), C, T, B, (uint64_t)C * 2,
                                (uint64_t)T * C * 2, 64, 128)) return 1;
        if (encode_tmap_bf16_3d(&maps.b[pl], plane(w, pl, (long long)k * 2 * C * C), C, (uint64_t)k * 2 * C, 1,
                                (uint64_t)C * 2, (uint64_t)k * 2 * C * C * 2, 64, 64)) return 1;
    }
    TcParams p = {};
    p.T = T; p.B = B; p.Kc = C; p.Nc = C; p.rows_per_tap = 2 * C; p.k = k; p.kb_n = C / 64;
    fill_taps_tc(p.tap_off, k, dilation, causal, false);
    p.bias = bias; p.spk = spk; p.res = res; p.y = y; p.save_a = save_a; p.save_s = save_s;
    p.gate_mode = mode; p.residual = residual;
    p.gmain = 1.f + config().tc_gamma * (float)(p.k * p.kb_n * 4);
    p.idesc_fmt = IDESC_A_F16 | IDESC_B_F16;                     // forward operands: fp16 hi/lo planes
    return launch_conv<TC_GATED, 2, 64, 64>(maps, p, t_tiles, C / 64, B, (cudaStream_t)stream, "tc_convblock_fwd");
}

// Generic conv / data-gradient:  out (B, Nc, T) fp32 = sum_j A[b, t+off_j, :] . W[j, n, :]  (+ epilogue)
//   a: [2][B][T][Kp] bf16 planes, Kp = Kc rounded up to 8;  w: [2][k][Nc][Kp] bf16 planes.
//   transpose_taps = 1 for a data gradient (offsets padl - j*d), 0 for a forward conv.
// Tile width: 128 output channels, or 64 when 128-wide tiles would leave most of the SMs idle.  BK = 64 needs
// Kc % 64 == 0 (else BK = 32: the 80-channel mel input, the 513-wide linear output, the 16-wide speaker embedding).
int dv3_tc_conv(const void* a, const void* w, int npl, float* out, int B, int Kc, int Nc, int T, int k, int dilation,
                int causal, int transpose_taps, const float* bias, int relu, float p_drop,
                const unsigned long long* seed_ptr, unsigned salt, int addmode, const float* e1, const float* e2,
                float alpha, const void* reserved, void* stream) {
    DV3_REQUIRE(reserved == nullptr, "tc_conv: reserved must be NULL");
    DV3_REQUIRE(k >= 1 && k <= MAX_TAPS_TC && (k == 1 || Nc % 128 == 0) && B <= 65535,
                "tc_conv: unsupported shape B=%d Kc=%d Nc=%d T=%d k=%d", B, Kc, Nc, T, k);
    DV3_REQUIRE(npl == 2, "tc_conv: npl must be 2");
    const int Kp = (Kc + 7) / 8 * 8;
    const int t_tiles = (T + 127) / 128;
    cudaStream_t st = (cudaStream_t)stream;
    const long long tiles128 = (long long)t_tiles * ((Nc + 127) / 128) * B;
    const bool narrow = Nc > 64 && (k == 1 || Nc % 64 == 0) && tiles128 < 100;
    const bool k64 = Kc % 64 == 0;
    const int bk = k64 ? 64 : 32, br = narrow ? 64 : 128;
    TcMaps maps;
    for (int pl = 0; pl < 2; ++pl) {
        if (encode_tmap_bf16_3d(&maps.a[pl], plane(a, pl, (long long)B * T * Kp), Kc, T, B, (uint64_t)Kp * 2,
                                (uint64_t)T * Kp * 2, bk, 128)) return 1;
        if (encode_tmap_bf16_3d(&maps.b[pl], plane(w, pl, (long long)k * Nc * Kp), Kc, (uint64_t)k * Nc, 1,
                                (uint64_t)Kp * 2, (uint64_t)k * Nc * Kp * 2, bk, br)) return 1;
    }
    TcParams p = {};
    p.T = T; p.B = B; p.Kc = Kc; p.Nc = Nc; p.rows_per_tap = Nc; p.k = k; p.kb_n = (Kc + bk - 1) / bk;
    fill_taps_tc(p.tap_off, k, dilation, causal, transpose_taps != 0);
    p.out = out; p.bias = bias; p.relu = relu; p.e1 = e1; p.e2 = e2; p.alpha = alpha; p.addmode = addmode;
    p.p_drop = p_drop; p.seed_ptr = seed_ptr; p.salt = salt;
    p.gmain = 1.f + config().tc_gamma * (float)(p.k * p.kb_n * (bk / 16));
    // forward conv: fp16 activation x fp16 weight planes; data gradient: bf16 gradient x bf16 weight planes
    p.idesc_fmt = transpose_taps ? (IDESC_A_BF16 | IDESC_B_BF16) : (IDESC_A_F16 | IDESC_B_F16);
    const int tiles_y = (Nc + br - 1) / br;
    if (narrow) {
        if (k64) return launch_conv<TC_CONV, 1, 64, 64>(maps, p, t_tiles, tiles_y, B, st, "tc_conv(64)");
        return launch_conv<TC_CONV, 1, 64, 32>(maps, p, t_tiles, tiles_y, B, st, "tc_conv(64,bk32)");
    }
    if (k64) return launch_conv<TC_CONV, 1, 128, 64>(maps, p, t_tiles, tiles_y, B, st, "tc_conv(128)");
    return launch_conv<TC_CONV, 1, 128, 32>(maps, p, t_tiles, tiles_y, B, st, "tc_conv(128,bk32)");
}

int dv3_tc_wgrad_nsplit(int B, int Mw, int Nw, int T, int k) {
    const int nt = Nw > 128 ? (Nw + 255) / 256 : 1;
    const int tiles = ((Mw + 127) / 128) * nt * k;
    // split (b,t) over enough CTAs for two waves, unless that leaves each CTA fewer than ~64 K-iterations (then the
    // per-CTA prologue/epilogue and the extra partial traffic cost more than the parallelism buys: one wave).
    // Measured on the preset shapes (tools/tc_time.py): (512,800) prefers 296, (256,800)/(512,128)/(256,200) prefer 148.
    const int kb_n = (T + 31) / 32;
    int best = 1;
    for (int target = 2 * 148; target >= 148; target -= 148) {
        int want = (target + tiles - 1) / tiles;
        if (want > B) want = B;
        if (want < 1) want = 1;
        const int bps = (B + want - 1) / want;
        best = (B + bps - 1) / bps;
        if (bps * kb_n >= 64) break;
    }
    return best;
}

// Weight gradient from (B,T,C) planes.  dy: [2][B][T][pad8(Mw)], xd: [2][B][T][pad8(Nw)]; partial element (m, n, j) at
// (m%msplit)*s_m + (m/msplit)*s_mh + n*s_n + j*s_j of split `s` at dw_partials + s*split_stride.
int dv3_tc_wgrad_mn(const void* dy, const void* xd, float* dw_partials, long long split_stride, int B, int Mw,
                    int Nw, int T, int k, int dilation, int causal, int msplit, long long s_m, long long s_mh,
                    long long s_n, long long s_j, void* stream) {
    DV3_REQUIRE(k >= 1 && k <= MAX_TAPS_TC && B <= 65535, "tc_wgrad_mn: unsupported shape k=%d", k);
    const int Mp = (Mw + 7) / 8 * 8, Np = (Nw + 7) / 8 * 8;
    TcMaps maps;
    for (int pl = 0; pl < 2; ++pl) {
        if (encode_tmap_bf16_3d(&maps.a[pl], plane(dy, pl, (long long)B * T * Mp), Mw, T, B, (uint64_t)Mp * 2,
                                (uint64_t)T * Mp * 2, 64, 32)) return 1;
        if (encode_tmap_bf16_3d(&maps.b[pl], plane(xd, pl, (long long)B * T * Np), Nw, T, B, (uint64_t)Np * 2,
                                (uint64_t)T * Np * 2, 64, 32)) return 1;
    }
    TcMnParams p = {};
    p.T = T; p.B = B; p.Mw = Mw; p.Nw = Nw; p.k = k; p.kb_n = (T + 31) / 32;
    fill_taps_tc(p.tap_off, k, dilation, causal, false);
    p.nsplit = dv3_tc_wgrad_nsplit(B, Mw, Nw, T, k);
    p.batches_per_split = (B + p.nsplit - 1) / p.nsplit;
    p.dw = dw_partials; p.split_stride = split_stride;
    p.msplit = msplit; p.s_m = s_m; p.s_mh = s_mh; p.s_n = s_n; p.s_j = s_j;
    p.gcoef = config().tc_gamma;
    cudaStream_t st = (cudaStream_t)stream;
    const int m_tiles = (Mw + 127) / 128;
    cudaError_t e;
    if (Nw > 128) {
        constexpr int SMEM = 4 * 2 * (2 * 4096 + 4 * 4096) + 1024 + 512;
        static const int configured = ensure_smem(tc_wgrad_mn_kernel<2>, SMEM, "tc_wgrad_mn");
        if (configured) return 1;
        e = launch_k(tc_wgrad_mn_kernel<2>, dim3((Nw + 255) / 256, m_tiles, p.nsplit * k), dim3(TC_THREADS), (size_t)SMEM,
                     st, maps, p);
    } else {
        constexpr int SMEM = 6 * 2 * (2 * 4096 + 2 * 4096) + 1024 + 512;
        static const int configured = ensure_smem(tc_wgrad_mn_kernel<1>, SMEM, "tc_wgrad_mn");
        if (configured) return 1;
        e = launch_k(tc_wgrad_mn_kernel<1>, dim3(1, m_tiles, p.nsplit * k), dim3(TC_THREADS), (size_t)SMEM, st, maps, p);
    }
    if (e != cudaSuccess) { set_error("tc_wgrad_mn: launch failed: %s", cudaGetErrorString(e)); return 1; }
    return check_launch("tc_wgrad_mn");
}

}  // extern "C"
