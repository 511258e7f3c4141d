// Fused dot-product attention of the teacher-forced decoder on tcgen05 tensor cores -- reference
// deepvoice3.py:132-176 (AttentionLayer.forward between the projections):
//     S = Q.K^T (no 1/sqrt(d)) -> mask padded keys with -inf -> softmax over keys -> [return P] -> dropout
//       -> O = scale * Pd.V                                                     (scale = Ts * sqrt(1/Ts))
// and its backward.  Layouts are the channel-major ones the decoder already holds: q (B,E,Td), k, v (B,E,Ts),
// out (B,E,Td), probabilities (B,Td,Ts) (materialised: the guided-attention loss reads them, train.py:734-738).
//
// Arithmetic: fp32-equivalent split-bf16 (hi*hi in one TMEM accumulator, hi*lo + lo*hi in a second one, summed in
// fp32 by the epilogue -- same scheme as tc_gemm.cu).  The fp32 operands are split INSIDE the kernel while they are
// staged into shared memory in the UMMA canonical layouts (there is no pre-pass and nothing but q/k/v/probs ever
// touches HBM):
//   * operands whose contraction index is the ROW of the global tensor (q, k, dO, v in the score GEMMs; P, dS in the
//     key/value-gradient GEMMs) are written MN-major: [contraction row][64 elements = 128 B], 16-byte chunk c of row
//     r at chunk position c ^ (r & 7) (SWIZZLE_128B), 64-element column groups LBO bytes apart;
//   * operands whose contraction index is contiguous in memory (v, k in the context GEMMs; dO, q in the gradient
//     GEMMs; the softmax output, produced by the epilogue threads themselves) are written K-major: [row][64
//     contraction elements = 128 B], 8-row atoms of 1024 B, same XOR swizzle.
//
// Kernels:
//   attn_rows_kernel<BWD=0>  one CTA per (128 query rows, utterance): S GEMM -> softmax epilogue (writes P, stages
//                            dropout(P) as the A operand of the second GEMM) -> O GEMM -> store.
//   attn_rows_kernel<BWD=1>  same skeleton for the backward: dPd = dO^T.V -> softmax backward epilogue (writes dS)
//                            -> dQ = dS.K^T.
//   attn_cols_kernel         one CTA per (128 channels, utterance): dV = scale * dO.Pd and dK = Q.dS, contraction over
//                            the query axis (which spans the CTAs of attn_rows_kernel, hence a second launch).
// 256 threads: all stage operands; thread 0 issues the MMAs; warps 0-3 (TMEM lane quarter = warp) run the epilogues.
#include "tc_common.cuh"

namespace dv3 {

using namespace tc;

constexpr int AT_THREADS = 256;
constexpr int AT_NS = 128;                 // key tile: Ts <= 128 (longer memories use the SIMT path)

struct AttnParams {
    const float* a1;        // rows kernel: q (fwd) / dO (bwd), (B,E,Td)
    const float* b1;        // rows kernel: k (fwd) / v (bwd), (B,E,Ts)
    const float* b2;        // rows kernel: v (fwd) / k (bwd), (B,E,Ts)
    const unsigned char* mask;   // (B,Ts) 1 = padding, or null (fwd)
    float* probs;           // (B,Td,Ts): written by fwd, read by bwd
    const float* dprobs;    // bwd: gradient arriving at the returned probabilities, or null
    float* ds;              // bwd: dS (B,Td,Ts) out (consumed by attn_cols_kernel)
    float* out;             // (B,E,Td): context (fwd) / dq (bwd)
    int B, E, Td, Ts;
    float scale, p_drop;
    const unsigned long long* seed_ptr;
    uint32_t salt;
};

__device__ __forceinline__ uint64_t desc_kmajor(uint32_t saddr) {            // [row][64 k] 128-byte rows, SWIZZLE_128B
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t saddr, uint32_t lbo) {   // [k row][64 mn], chunk stride lbo
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// 8 fp32 -> 8 bf16 hi (16 bytes) + 8 bf16 lo
__device__ __forceinline__ void split8(const float* x, uint4& hi, uint4& lo) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat16 h0 = __float2bfloat16_rn(x[2 * i]), h1 = __float2bfloat16_rn(x[2 * i + 1]);
        const __nv_bfloat16 l0 = __float2bfloat16_rn(x[2 * i] - __bfloat162float(h0));
        const __nv_bfloat16 l1 = __float2bfloat16_rn(x[2 * i + 1] - __bfloat162float(h1));
        h[i] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        l[i] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// 8 consecutive floats row[c0 .. c0+8) with bounds (cols >= ncols read as 0); vectorised when aligned
__device__ __forceinline__ void load8(const float* __restrict__ row, int c0, int ncols, bool row_ok, bool vec_ok,
                                      float* x) {
    if (row_ok && vec_ok && c0 + 8 <= ncols) {
        const float4 u = __ldg(reinterpret_cast<const float4*>(row + c0));
        const float4 w = __ldg(reinterpret_cast<const float4*>(row + c0 + 4));
        x[0] = u.x; x[1] = u.y; x[2] = u.z; x[3] = u.w; x[4] = w.x; x[5] = w.y; x[6] = w.z; x[7] = w.w;
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = (row_ok && c0 + i < ncols) ? __ldg(row + c0 + i) : 0.f;
    }
}

// The staging loops below issue the global loads of UNR groups (2 x float4 each) before the first conversion / shared
// store, so a thread has UNR x 32 bytes in flight instead of one group (the one-group-at-a-time version was latency
// bound: 60-140 us per launch for ~1 MB of operands).
constexpr int ST_UNR = 4;

// Stage an MN-major operand chunk: 64 contraction rows (global rows r0 .. r0+64 of a (nrows, ncols) matrix, row stride
// ld) x NCH*64 columns starting at column c_base; two planes (hi at dst, lo at dst + plane_bytes); chunk stride 8 KB.
template <int NCH>
__device__ __forceinline__ void stage_mn(uint8_t* dst, uint32_t plane_bytes, const float* __restrict__ src, long long ld,
                                         int r0, int nrows, int c_base, int ncols, bool vec_ok, int tid, int nthreads) {
    constexpr int GROUPS_PER_ROW = NCH * 8;                // 16-byte chunks (8 elements) per row
    constexpr int TOTAL = 64 * GROUPS_PER_ROW;
    for (int g0 = tid; g0 < TOTAL; g0 += nthreads * ST_UNR) {
        float x[ST_UNR][8];
#pragma unroll
        for (int u = 0; u < ST_UNR; ++u) {
            const int g = g0 + u * nthreads;
            const int r = g / GROUPS_PER_ROW, cg = g - r * GROUPS_PER_ROW;
            load8(src + (long long)(r0 + r) * ld, c_base + cg * 8, ncols, g < TOTAL && r0 + r < nrows, vec_ok, x[u]);
        }
#pragma unroll
        for (int u = 0; u < ST_UNR; ++u) {
            const int g = g0 + u * nthreads;
            if (g >= TOTAL) break;
            const int r = g / GROUPS_PER_ROW, cg = g - r * GROUPS_PER_ROW;
            const int h = cg >> 3, c = cg & 7;
            uint4 hi, lo;
            split8(x[u], hi, lo);
            const uint32_t off = (uint32_t)h * 8192u + (uint32_t)r * 128u + (uint32_t)((c ^ (r & 7)) << 4);
            *reinterpret_cast<uint4*>(dst + off) = hi;
            *reinterpret_cast<uint4*>(dst + plane_bytes + off) = lo;
        }
    }
}

// Stage a K-major operand: nrows_tile rows (global rows r0.., row stride ld) x 64 contraction columns starting at c_base.
__device__ __forceinline__ void stage_k(uint8_t* dst, uint32_t plane_bytes, const float* __restrict__ src, long long ld,
                                        int r0, int nrows_valid, int nrows_tile, int c_base, int ncols, bool vec_ok,
                                        int tid, int nthreads) {
    const int total = nrows_tile * 8;
    for (int g0 = tid; g0 < total; g0 += nthreads * ST_UNR) {
        float x[ST_UNR][8];
#pragma unroll
        for (int u = 0; u < ST_UNR; ++u) {
            const int g = g0 + u * nthreads;
            const int r = g >> 3, c = g & 7;
            load8(src + (long long)(r0 + r) * ld, c_base + c * 8, ncols, g < total && r0 + r < nrows_valid, vec_ok, x[u]);
        }
#pragma unroll
        for (int u = 0; u < ST_UNR; ++u) {
            const int g = g0 + u * nthreads;
            if (g >= total) break;
            const int r = g >> 3, c = g & 7;
            uint4 hi, lo;
            split8(x[u], hi, lo);
            const uint32_t off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u + (uint32_t)((c ^ (r & 7)) << 4);
            *reinterpret_cast<uint4*>(dst + off) = hi;
            *reinterpret_cast<uint4*>(dst + plane_bytes + off) = lo;
        }
    }
}

__device__ __forceinline__ void tmem_ld_sum(uint32_t taddr, int cross_off, float* v) {
    float c[32];
    tmem_ld_32x32(taddr, v);
    tmem_ld_32x32(taddr + cross_off, c);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] += c[i];
}

// main (+)= Ahi*Bhi ; cross (+)= Ahi*Blo + Alo*Bhi
__device__ __forceinline__ void mma3(uint32_t tmain, uint32_t tcross, uint64_t ahi, uint64_t alo, uint64_t bhi,
                                     uint64_t blo, uint32_t idesc, bool first) {
    umma_bf16(tmain, ahi, bhi, idesc, first ? 0u : 1u);
    umma_bf16(tcross, ahi, blo, idesc, first ? 0u : 1u);
    umma_bf16(tcross, alo, bhi, idesc, 1u);
}

// Shared-memory map of attn_rows_kernel (bytes, after 1024-byte alignment):
//   phase 1 (two stages of 64 KB):  stage s at s*65536: A hi 16 KB | A lo 16 KB | B hi 16 KB | B lo 16 KB
//   phase 2 (aliases phase 1):      A2 hi 32 KB | A2 lo 32 KB  (2 key slabs x 128 rows x 128 B)
//                                   B2 at 65536: per key slab [hi E*128 | lo E*128]  (<= 2 x 64 KB)
// Epilogue warps exchange 32 x 32 tiles with global memory through a per-warp transposing buffer: the thread of TMEM
// lane r owns ROW r of the score tile, and a row of the (B,Td,Ts) probability tensors is contiguous along the keys -- a
// direct per-thread access touches 32 different 128-byte lines per warp instruction (ncu: the softmax epilogues were
// bound by those LSU transactions).  Through the buffer every global access is one full 128-byte line per instruction.
constexpr int TILE_PITCH = 33;
constexpr int TILE_FLOATS = 32 * TILE_PITCH;
constexpr int ROWS_SMEM = 65536 + 2 * 65536 + 1024 + 256 + 4 * TILE_FLOATS * 4;

// global rows [0, rows_valid) x columns [c0, c0+32) of a row-major matrix (row stride ld) starting at src -> tile
__device__ __forceinline__ void tile_load(float* tile, const float* __restrict__ src, int ld, int rows_valid, int c0,
                                          int ncols, int lane) {
    __syncwarp();
    const bool cok = c0 + lane < ncols;
#pragma unroll 8
    for (int rr = 0; rr < 32; ++rr)
        tile[rr * TILE_PITCH + lane] = (cok && rr < rows_valid) ? __ldg(src + (size_t)rr * ld + c0 + lane) : 0.f;
    __syncwarp();
}
// tile -> global rows [0, rows_valid) x columns [c0, c0+32)
__device__ __forceinline__ void tile_store(const float* tile, float* __restrict__ dst, int ld, int rows_valid, int c0,
                                           int ncols, int lane) {
    __syncwarp();
    const bool cok = c0 + lane < ncols;
#pragma unroll 8
    for (int rr = 0; rr < 32; ++rr)
        if (cok && rr < rows_valid) dst[(size_t)rr * ld + c0 + lane] = tile[rr * TILE_PITCH + lane];
    __syncwarp();
}

template <int BWD>
__global__ void __launch_bounds__(AT_THREADS, 1) attn_rows_kernel(const __grid_constant__ AttnParams p) {
    pdl_trigger();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 3 * 65536);        // [0,1]: stage free, [2]: GEMM1 done, [3]: GEMM2 done
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 4);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y, t0 = blockIdx.x * 128;
    const int E = p.E, Td = p.Td, Ts = p.Ts;
    const float* A1 = p.a1 + (size_t)b * E * Td;
    const float* B1 = p.b1 + (size_t)b * E * Ts;
    const float* B2 = p.b2 + (size_t)b * E * Ts;
    const bool vec_td = (Td & 3) == 0, vec_ts = (Ts & 3) == 0;

    if (tid == 0) {
        for (int i = 0; i < 4; ++i) mbar_init(&bars[i], 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc<512>(tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_ptr;
    pdl_wait();                 // set-up above overlaps the previous kernel's tail; global memory from here on

    // ---------------- GEMM 1: D1[t][s] = sum_e A1[e][t0+t] * B1[e][s] -----------------------------------
    const int kchunks = (E + 63) / 64;
    constexpr uint32_t idesc_mn = make_idesc_bf16(128, AT_NS) | (1u << 15) | (1u << 16);
    for (int kc = 0; kc < kchunks; ++kc) {
        const int s = kc & 1;
        if (kc >= 2) mbar_wait(&bars[s], ((kc >> 1) - 1) & 1);          // the MMAs that read this stage retired
        uint8_t* st = smem + s * 65536;
        stage_mn<2>(st, 16384, A1, Td, kc * 64, E, t0, Td, vec_td, tid, AT_THREADS);
        stage_mn<2>(st + 32768, 16384, B1, Ts, kc * 64, E, 0, Ts, vec_ts, tid, AT_THREADS);
        fence_proxy_async();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            const uint32_t sa = smem_u32(st);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const uint32_t ko = kk * 2048;
                mma3(tmem, tmem + AT_NS, desc_mnmajor(sa + ko, 8192), desc_mnmajor(sa + 16384 + ko, 8192),
                     desc_mnmajor(sa + 32768 + ko, 8192), desc_mnmajor(sa + 49152 + ko, 8192), idesc_mn,
                     kc == 0 && kk == 0);
            }
            umma_commit(&bars[s]);
            if (kc == kchunks - 1) umma_commit(&bars[2]);
        }
    }
    mbar_wait(&bars[2], 0);
    tc_fence_after();

    // ---------------- epilogue 1 (warps 0-3) || stage B2 (warps 4-7) -------------------------------------
    const int nslab = (Ts + 63) / 64;                       // 64-key slabs of the second contraction
    const uint32_t b2_plane = (uint32_t)E * 128u;           // one plane of one slab: E rows x 128 B
    if (warp >= 4) {
        for (int sl = 0; sl < nslab; ++sl)
            stage_k(smem + 65536 + sl * 2 * b2_plane, b2_plane, B2, Ts, 0, E, E, sl * 64, Ts, vec_ts, tid - 128, 128);
    } else {
        const int row = warp * 32 + lane, t = t0 + row;
        const bool tv = t < Td;
        const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
        const DropCfg drop = make_drop(p.p_drop, p.seed_ptr, p.salt);
        const size_t rbase = ((size_t)b * Td + (tv ? t : 0)) * Ts;
        const unsigned char* mrow = p.mask ? p.mask + (size_t)b * Ts : nullptr;
        // this warp's 32 rows of the (B,Td,Ts) tensors, accessed through the transposing tile (see TILE_PITCH)
        float* tile = reinterpret_cast<float*>(smem + 3 * 65536 + 256) + warp * TILE_FLOATS;
        const int tw0 = t0 + warp * 32, rows_valid = min(max(Td - tw0, 0), 32);
        const size_t wbase = ((size_t)b * Td + min(tw0, Td - 1)) * Ts;
        float r0v = 0.f, r1v = 0.f;      // fwd: row max, 1/sum ; bwd: dot
        // key s is excluded (padding or beyond Ts) <=> bit (s & 31) of mb[s >> 5]: one byte load per lane and chunk
        uint32_t mb[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int s = 32 * j + lane;
            mb[j] = __ballot_sync(0xffffffffu, s >= Ts || (mrow && mrow[s < Ts ? s : 0]));
        }
        if (BWD == 0) {
            float mx = -INFINITY;
#pragma unroll
            for (int c32 = 0; c32 < AT_NS; c32 += 32) {
                float v[32];
                tmem_ld_sum(taddr + c32, AT_NS, v);
#pragma unroll
                for (int i = 0; i < 32; ++i) mx = fmaxf(mx, ((mb[c32 >> 5] >> i) & 1u) ? -INFINITY : v[i]);
            }
            float sum = 0.f;
#pragma unroll
            for (int c32 = 0; c32 < AT_NS; c32 += 32) {
                float v[32];
                tmem_ld_sum(taddr + c32, AT_NS, v);
#pragma unroll
                for (int i = 0; i < 32; ++i) sum += ((mb[c32 >> 5] >> i) & 1u) ? 0.f : expf(v[i] - mx);
            }
            r0v = mx; r1v = 1.f / sum;
        } else {
            float dot = 0.f;
            for (int c32 = 0; c32 < AT_NS; c32 += 32) {
                float v[32], pv[32];
                tmem_ld_sum(taddr + c32, AT_NS, v);
                if (c32 >= Ts) continue;                          // uniform
                tile_load(tile, p.probs + wbase, Ts, rows_valid, c32, Ts, lane);
#pragma unroll
                for (int i = 0; i < 32; ++i) pv[i] = tile[lane * TILE_PITCH + i];
                if (p.dprobs) tile_load(tile, p.dprobs + wbase, Ts, rows_valid, c32, Ts, lane);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int s = c32 + i;
                    if (tv && s < Ts) {
                        float g = p.scale * v[i] * drop_scale(drop, (uint32_t)(rbase + s));
                        if (p.dprobs) g += tile[lane * TILE_PITCH + i];
                        dot = fmaf(g, pv[i], dot);
                    }
                }
            }
            r0v = dot;
        }
        // probability of a masked key: 0, but NaN in a row whose keys are all masked (max -inf), which has no softmax
        // -- the SIMT kernel and torch's softmax of a row of -inf give NaN there too
        const float pr_masked = (BWD == 0 && r0v == -INFINITY) ? __int_as_float(0x7fc00000) : 0.f;
        // final pass: produce the row of the second GEMM's A operand (dropout(P) or dS), write P / dS to HBM
        for (int c32 = 0; c32 < AT_NS; c32 += 32) {
            float v[32], o[32];
            tmem_ld_sum(taddr + c32, AT_NS, v);
            const bool live = c32 < Ts;                           // uniform: chunks past the last key hold nothing
            const uint32_t mbc = c32 == 0 ? mb[0] : (c32 == 32 ? mb[1] : (c32 == 64 ? mb[2] : mb[3]));
            float pv[32];
            if (BWD == 1 && live) {
                tile_load(tile, p.probs + wbase, Ts, rows_valid, c32, Ts, lane);
#pragma unroll
                for (int i = 0; i < 32; ++i) pv[i] = tile[lane * TILE_PITCH + i];
                if (p.dprobs) tile_load(tile, p.dprobs + wbase, Ts, rows_valid, c32, Ts, lane);
            }
            float gp[32];                                         // fwd: the probability; bwd: dS
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int s = c32 + i;
                float a2 = 0.f, wr = 0.f;
                if (tv && s < Ts) {
                    if (BWD == 0) {
                        const bool ok = !((mbc >> i) & 1u);
                        const float pr = ok ? expf(v[i] - r0v) * r1v : pr_masked;
                        wr = pr;
                        a2 = pr * drop_scale(drop, (uint32_t)(rbase + s));
                    } else {
                        float g = p.scale * v[i] * drop_scale(drop, (uint32_t)(rbase + s));
                        if (p.dprobs) g += tile[lane * TILE_PITCH + i];
                        a2 = pv[i] * (g - r0v);
                        wr = a2;
                    }
                }
                o[i] = a2; gp[i] = wr;
            }
            if (live) {
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 32; ++i) tile[lane * TILE_PITCH + i] = gp[i];
                tile_store(tile, (BWD == 0 ? p.probs : p.ds) + wbase, Ts, rows_valid, c32, Ts, lane);
            }
            if (c32 < nslab * 64) {
#pragma unroll
                for (int c8 = 0; c8 < 4; ++c8) {
                    uint4 hi, lo;
                    split8(o + c8 * 8, hi, lo);
                    const int s = c32 + c8 * 8, sl = s >> 6, c = (s & 63) >> 3;
                    const uint32_t off = (uint32_t)sl * 16384u + (uint32_t)(row >> 3) * 1024u + (uint32_t)(row & 7) * 128u +
                                         (uint32_t)((c ^ (row & 7)) << 4);
                    *reinterpret_cast<uint4*>(smem + off) = hi;
                    *reinterpret_cast<uint4*>(smem + 32768 + off) = lo;
                }
            }
        }
        tc_fence_before();
    }
    fence_proxy_async();
    __syncthreads();

    // ---------------- GEMM 2: D2[t][e] = sum_s A2[t][s] * B2[e][s] ---------------------------------------
    if (tid == 0) {
        tc_fence_after();
        const uint32_t idesc_k = make_idesc_bf16(128, E);
        const uint32_t sa = smem_u32(smem), sb = smem_u32(smem + 65536);
        for (int sl = 0; sl < nslab; ++sl) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const uint32_t a_hi = sa + sl * 16384 + kk * 32, b_hi = sb + sl * 2 * b2_plane + kk * 32;
                mma3(tmem, tmem + 256, desc_kmajor(a_hi), desc_kmajor(a_hi + 32768), desc_kmajor(b_hi),
                     desc_kmajor(b_hi + b2_plane), idesc_k, sl == 0 && kk == 0);
            }
        }
        umma_commit(&bars[3]);
    }
    mbar_wait(&bars[3], 0);
    tc_fence_after();
    if (warp < 4) {
        const int row = warp * 32 + lane, t = t0 + row;
        const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
        const float sc = BWD == 0 ? p.scale : 1.f;
        float* __restrict__ out = p.out + (size_t)b * E * Td;
        for (int c32 = 0; c32 < E; c32 += 32) {             // E % 16 == 0: the last chunk may be half used
            float v[32];
            tmem_ld_sum(taddr + c32, 256, v);
            if (t < Td) {
#pragma unroll
                for (int i = 0; i < 32; ++i)
                    if (c32 + i < E) out[(size_t)(c32 + i) * Td + t] = sc * v[i];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem);
}

// dV[e][s] = scale * sum_t dO[e][t] * Pd[t][s] ;  dK[e][s] = sum_t Q[e][t] * dS[t][s]
// smem per 64-query chunk: A(dO) hi 16 KB | lo 16 KB | A(q) hi | lo | B(Pd) hi 16 KB | lo | B(dS) hi | lo  = 128 KB
constexpr int COLS_SMEM = 131072 + 1024 + 256;

struct AttnColsParams {
    const float* dout; const float* q; const float* probs; const float* ds;
    float* dv; float* dk;
    int B, E, Td, Ts;
    float scale, p_drop;
    const unsigned long long* seed_ptr;
    uint32_t salt;
};

__global__ void __launch_bounds__(AT_THREADS, 1) attn_cols_kernel(const __grid_constant__ AttnColsParams p) {
    pdl_trigger();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 131072);            // [0]: chunk MMAs retired
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y, e0 = blockIdx.x * 128;
    const int E = p.E, Td = p.Td, Ts = p.Ts;
    const float* dO = p.dout + (size_t)b * E * Td;
    const float* Q = p.q + (size_t)b * E * Td;
    const float* P = p.probs + (size_t)b * Td * Ts;
    const float* dS = p.ds + (size_t)b * Td * Ts;
    const bool vec_td = (Td & 3) == 0, vec_ts = (Ts & 3) == 0;
    const DropCfg drop = make_drop(p.p_drop, p.seed_ptr, p.salt);

    if (tid == 0) { mbar_init(&bars[0], 1); fence_barrier_init(); }
    if (warp == 0) tmem_alloc<512>(tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_ptr;
    pdl_wait();                 // set-up above overlaps the previous kernel's tail; global memory from here on

    const int kchunks = (Td + 63) / 64;
    constexpr uint32_t idesc = make_idesc_bf16(128, AT_NS) | (1u << 16);      // A K-major, B MN-major
    for (int kc = 0; kc < kchunks; ++kc) {
        if (kc >= 1) mbar_wait(&bars[0], (kc - 1) & 1);
        // A operands: rows e0.. of (E,Td), 64 query columns
        stage_k(smem, 16384, dO, Td, e0, E, 128, kc * 64, Td, vec_td, tid, AT_THREADS);
        stage_k(smem + 32768, 16384, Q, Td, e0, E, 128, kc * 64, Td, vec_td, tid, AT_THREADS);
        // B operands: 64 query rows of (Td,Ts); Pd = P * dropout mask regenerated from the element index
        {
            uint8_t* dst = smem + 65536;
            for (int g0 = tid; g0 < 64 * 16; g0 += AT_THREADS * 2) {
                float x[2][8], y[2][8];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int g = g0 + u * AT_THREADS, r = g >> 4, cg = g & 15, t = kc * 64 + r;
                    load8(P + (long long)t * Ts, cg * 8, Ts, t < Td, vec_ts, x[u]);
                    load8(dS + (long long)t * Ts, cg * 8, Ts, t < Td, vec_ts, y[u]);
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int g = g0 + u * AT_THREADS, r = g >> 4, cg = g & 15, h = cg >> 3, c = cg & 7;
                    const int t = kc * 64 + r;
                    if (drop.on) {
                        const size_t idx0 = ((size_t)b * Td + t) * Ts + cg * 8;
#pragma unroll
                        for (int i = 0; i < 8; ++i) x[u][i] *= drop_scale(drop, (uint32_t)(idx0 + i));
                    }
                    uint4 hi, lo;
                    const uint32_t off = (uint32_t)h * 8192u + (uint32_t)r * 128u + (uint32_t)((c ^ (r & 7)) << 4);
                    split8(x[u], hi, lo);
                    *reinterpret_cast<uint4*>(dst + off) = hi;
                    *reinterpret_cast<uint4*>(dst + 16384 + off) = lo;
                    split8(y[u], hi, lo);
                    *reinterpret_cast<uint4*>(dst + 32768 + off) = hi;
                    *reinterpret_cast<uint4*>(dst + 49152 + off) = lo;
                }
            }
        }
        fence_proxy_async();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            const uint32_t sa = smem_u32(smem);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const uint32_t ak = kk * 32, bk = kk * 2048;
                // dV: A = dO, B = Pd
                mma3(tmem, tmem + 128, desc_kmajor(sa + ak), desc_kmajor(sa + 16384 + ak),
                     desc_mnmajor(sa + 65536 + bk, 8192), desc_mnmajor(sa + 81920 + bk, 8192), idesc, kc == 0 && kk == 0);
                // dK: A = q, B = dS
                mma3(tmem + 256, tmem + 384, desc_kmajor(sa + 32768 + ak), desc_kmajor(sa + 49152 + ak),
                     desc_mnmajor(sa + 98304 + bk, 8192), desc_mnmajor(sa + 114688 + bk, 8192), idesc,
                     kc == 0 && kk == 0);
            }
            umma_commit(&bars[0]);
        }
    }
    mbar_wait(&bars[0], (kchunks - 1) & 1);
    tc_fence_after();
    if (warp < 4) {
        // rows e of dV / dK are contiguous along the keys: through the transposing tile (the operand buffers are free)
        const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
        float* tile = reinterpret_cast<float*>(smem) + warp * TILE_FLOATS;
        const int ew0 = e0 + warp * 32, rows_valid = min(max(E - ew0, 0), 32);
        const size_t wbase = ((size_t)b * E + min(ew0, E - 1)) * Ts;
        for (int c32 = 0; c32 < AT_NS; c32 += 32) {
            float v[32], w[32];
            tmem_ld_sum(taddr + c32, 128, v);
            tmem_ld_sum(taddr + 256 + c32, 128, w);
            if (c32 >= Ts) continue;                              // uniform
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 32; ++i) tile[lane * TILE_PITCH + i] = p.scale * v[i];
            tile_store(tile, p.dv + wbase, Ts, rows_valid, c32, Ts, lane);
#pragma unroll
            for (int i = 0; i < 32; ++i) tile[lane * TILE_PITCH + i] = w[i];
            tile_store(tile, p.dk + wbase, Ts, rows_valid, c32, Ts, lane);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem);
}

template <typename K>
static int set_smem(K kern, int bytes, const char* what) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) { set_error("%s: cannot set %d B dynamic smem: %s", what, bytes, cudaGetErrorString(e)); return 1; }
    return 0;
}

}  // namespace dv3

using namespace dv3;

extern "C" {

// 1 if the tensor-core attention kernels cover this shape (else the caller uses dv3_bgemm + dv3_softmax_*)
int dv3_tc_attn_supported(int B, int E, int Td, int Ts) {
    return B >= 1 && B <= 65535 && E >= 16 && E <= 256 && (E % 16) == 0 && Ts >= 1 && Ts <= AT_NS && Td >= 1;
}

int dv3_tc_attn_fwd(const float* q, const float* k, const float* v, const unsigned char* mask, float* probs,
                    float* out, int B, int E, int Td, int Ts, float scale, float p_drop,
                    const unsigned long long* seed_ptr, unsigned salt, void* stream) {
    DV3_REQUIRE(dv3_tc_attn_supported(B, E, Td, Ts), "tc_attn_fwd: unsupported shape B=%d E=%d Td=%d Ts=%d", B, E, Td, Ts);
    static bool configured = false;
    if (!configured) { if (set_smem(attn_rows_kernel<0>, ROWS_SMEM, "tc_attn_fwd")) return 1; configured = true; }
    AttnParams p = {};
    p.a1 = q; p.b1 = k; p.b2 = v; p.mask = mask; p.probs = probs; p.out = out;
    p.B = B; p.E = E; p.Td = Td; p.Ts = Ts; p.scale = scale; p.p_drop = p_drop; p.seed_ptr = seed_ptr; p.salt = salt;
    launch_k(attn_rows_kernel<0>, dim3((Td + 127) / 128, B), AT_THREADS, ROWS_SMEM, (cudaStream_t)stream, p);
    return check_launch("tc_attn_fwd");
}

// ds: scratch (B,Td,Ts) fp32 written by the first launch and read by the second; dprobs may be null
int dv3_tc_attn_bwd(const float* dout, const float* q, const float* k, const float* v, const float* probs,
                    const float* dprobs, float* ds, float* dq, float* dk, float* dv, int B, int E, int Td, int Ts,
                    float scale, float p_drop, const unsigned long long* seed_ptr, unsigned salt, void* stream) {
    DV3_REQUIRE(dv3_tc_attn_supported(B, E, Td, Ts), "tc_attn_bwd: unsupported shape B=%d E=%d Td=%d Ts=%d", B, E, Td, Ts);
    static bool configured = false;
    if (!configured) {
        if (set_smem(attn_rows_kernel<1>, ROWS_SMEM, "tc_attn_bwd")) return 1;
        if (set_smem(attn_cols_kernel, COLS_SMEM, "tc_attn_bwd")) return 1;
        configured = true;
    }
    AttnParams p = {};
    p.a1 = dout; p.b1 = v; p.b2 = k; p.probs = const_cast<float*>(probs); p.dprobs = dprobs; p.ds = ds; p.out = dq;
    p.B = B; p.E = E; p.Td = Td; p.Ts = Ts; p.scale = scale; p.p_drop = p_drop; p.seed_ptr = seed_ptr; p.salt = salt;
    launch_k(attn_rows_kernel<1>, dim3((Td + 127) / 128, B), AT_THREADS, ROWS_SMEM, (cudaStream_t)stream, p);
    if (check_launch("tc_attn_bwd(rows)")) return 1;
    AttnColsParams c = {};
    c.dout = dout; c.q = q; c.probs = probs; c.ds = ds; c.dv = dv; c.dk = dk;
    c.B = B; c.E = E; c.Td = Td; c.Ts = Ts; c.scale = scale; c.p_drop = p_drop; c.seed_ptr = seed_ptr; c.salt = salt;
    launch_k(attn_cols_kernel, dim3((E + 127) / 128, B), AT_THREADS, COLS_SMEM, (cudaStream_t)stream, c);
    return check_launch("tc_attn_bwd(cols)");
}

}  // extern "C"
