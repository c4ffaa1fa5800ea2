// Kernel 3c -- a whole SLOTS set-abstraction level in ONE launch (included by sa_tc.cu).
//
//   gather + concat -> MMA1 -> epilogue (affine + ReLU) -> shared memory -> MMA2 -> epilogue -> shared memory -> MMA3 ->
//   per-centroid max
//
// i.e. PointNetConv(local_nn) of /root/reference/pointnet2_regressor.py:18 with BatchNorm in EVALUATION mode (running
// statistics: the reference's test-time pass, /root/reference/testing_model.py:56-64): nothing but the [n_dst, c3] output
// ever leaves the SM.  The multi-pass kernels of sa_tc.cu stored every hidden activation twice (zhat and a) and made five
// GEMM passes per level because train-mode BatchNorm needs batch statistics between the layers; evaluation does not.
//
// Work unit: a tile of 64 compacted rows (a centroid never crosses a 64-row boundary), channels on the TMEM lanes, rows
// on the TMEM columns (UMMA M = 128, N = 64) -- the orientation of every kernel here, so the per-centroid max is again a
// per-thread scan of accumulator columns.  A CTA keeps TWO tiles in flight (slots): each slot has its own loader warps,
// epilogue warps, shared-memory operand buffers and TMEM columns, one thread issues the MMAs of both.  All three weight
// images stay resident in shared memory.
//
//   warps  0- 7 / 8-15   epilogue group of slot 0 / 1: warp w drains TMEM lane quarter w % 4, column half (w / 4) % 2
//   warps 16 / 17        MMA issuer of slot 0 / 1 (warp 16 owns the TMEM allocation).  The WHOLE warp runs the issue loop and
//                        one elected lane executes the tcgen05 instructions: under a divergent `if (lane == 0)` every
//                        operand descriptor went through R2UR moves (4-5 per tcgen05.mma, ncu round 2); warp-uniform code
//                        keeps them in uniform registers
//   warps 18-21 / 22-25  gather loaders of slot 0 / 1: two threads per row of the tile; the row indices of the NEXT tile are
//                        prefetched and all loads of a row are in flight together (the gather is a chain of dependent
//                        L2 round trips: row -> source index -> feature row)
//
// Shared-memory operand tiles follow tc_common.cuh: 128-byte lines, SWIZZLE_128B.  The gathered layer-1 operand is a K-major
// B tile (line = row); the epilogues write the next layer's operand as an MN-major B tile (line = channel, 64 rows per line).
#pragma once

namespace b2pn {
namespace tc {

constexpr int CH_ROWS = 64;
constexpr int CH_SLOTS = 2;
constexpr int CH_EPI_WARPS = 8;                       // per slot
constexpr int CH_EPI_THREADS = CH_EPI_WARPS * 32;     // 256
constexpr int CH_LOAD_THREADS = 128;                  // per slot: two threads per row of the tile
constexpr int CH_MMA_WARP = CH_SLOTS * CH_EPI_WARPS;  // 16, 17: one MMA issuer warp per slot
constexpr int CH_THREADS = CH_SLOTS * CH_EPI_THREADS + CH_SLOTS * 32 + CH_SLOTS * CH_LOAD_THREADS;  // 832
constexpr int CH_CHUNK_BYTES = CH_ROWS * LINE_BYTES;  // 8 KB: 64 rows x 64 k (K-major) or 64 channel lines x 64 rows (MN-major)
constexpr int CH_TMEM_PER_SLOT = 256;                 // D1 [0,64) D2 [64,128) D3 [128, 128 + 64 mt3)

struct ChainParams {
    const uint8_t *w_img[3];  // fp16 weight images (pack_weights_kernel), num_mg == 1
    int w_bytes[3];
    int k_img;                // real columns of the layer-1 operand
    int k1c, c1c, c2c;        // K chunks (of 64) of layers 1, 2, 3
    int c1, c2, c3;           // channels
    int mt3;                  // M tiles of layer 3 (1: c3 <= 128, 2: c3 <= 256)
    int64_t rows;
    const int64_t *rows_dev;
    // evaluation-mode BatchNorm folded into one multiply-add per element: y = act(acc * scale + shift)
    const float *bias[3];
    const float *gamma[2], *beta[2], *mean[2], *var[2];
    float eps;
    int act;
    float *out;               // [n_dst][c3]
    int32_t *arg;             // [n_dst][c3] arg-max slot
    __half *out16;            // optional fp16 copy of out
    const uint32_t *rgrp;
};

// barriers of a slot
enum { CB_B1_FULL = 0, CB_B1_FREE, CB_D1_FULL, CB_A1_FULL, CB_D2_FULL, CB_A2_FULL, CB_D3_FULL, CB_D3_FREE, CB_PER_SLOT };

__device__ __forceinline__ void chain_affine(const ChainParams &p, int layer, int ch, float &scale, float &shift)
{
    scale = 0.f;
    shift = 0.f;
    const int C = layer == 0 ? p.c1 : p.c2;
    if (ch < C) {
        const float rstd = 1.0f / sqrtf(p.var[layer][ch] + p.eps);
        scale = p.gamma[layer][ch] * rstd;
        shift = fmaf(p.bias[layer][ch] - p.mean[layer][ch], scale, p.beta[layer][ch]);
    }
}

// Shape parameters as template arguments (-1: take the run-time value of ChainParams).  The MMA issuer is ONE thread: with
// run-time loop bounds its descriptor arithmetic is a dependent instruction stream of ~20 instructions per tcgen05.mma at
// 4-6 cycles each, which made every MMA hop of the chain ~2000 cycles long (ncu, round 2: the epilogue warps spent 55 % of
// their time waiting for D2 / D3); fully unrolled, a tcgen05.mma costs two 64-bit adds.
template <int K1C_, int NKS_LAST_, int C1C_, int C2C_, int MT3_>
__global__ void __launch_bounds__(CH_THREADS, 1) tc_chain_eval_kernel(const ChainParams p, GatherLoaderTC gl)
{
    const int k1c = K1C_ >= 0 ? K1C_ : p.k1c;
    const int c1c = C1C_ >= 0 ? C1C_ : p.c1c;
    const int c2c = C2C_ >= 0 ? C2C_ : p.c2c;
    const int mt3 = MT3_ >= 0 ? MT3_ : p.mt3;
    const int nks_last = NKS_LAST_ >= 0 ? NKS_LAST_ : ((p.k_img - (p.k1c - 1) * KC) >= KC ? 4 : (p.k_img - (p.k1c - 1) * KC + 15) / 16);
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *W0 = smem, *W1 = W0 + p.w_bytes[0], *W2 = W1 + p.w_bytes[1];
    uint8_t *slots = W2 + p.w_bytes[2];
    const int b1_bytes = k1c * CH_CHUNK_BYTES;
    const int x_bytes = (c1c > c2c ? c1c : c2c) * CH_CHUNK_BYTES;
    const int slot_bytes = b1_bytes + x_bytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(slots + CH_SLOTS * slot_bytes);
    uint64_t *w_full = bars + CH_SLOTS * CB_PER_SLOT;
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(w_full + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t rows = p.rows_dev ? *p.rows_dev : p.rows;
    const int64_t num_tiles = (rows + CH_ROWS - 1) / CH_ROWS;
    gl.resolve(rows);

    if (tid == 0) {
        for (int s = 0; s < CH_SLOTS; ++s) {
            uint64_t *b = bars + s * CB_PER_SLOT;
            // one arrival per WARP (its lanes fence their own writes, __syncwarp, lane 0 arrives): 256 arrivals on one
            // shared-memory word would serialise for ~250 cycles per barrier
            mbar_init(&b[CB_B1_FULL], CH_LOAD_THREADS / 32);
            mbar_init(&b[CB_B1_FREE], 1);
            mbar_init(&b[CB_D1_FULL], 1);
            mbar_init(&b[CB_A1_FULL], CH_EPI_WARPS);
            mbar_init(&b[CB_D2_FULL], 1);
            mbar_init(&b[CB_A2_FULL], CH_EPI_WARPS);
            mbar_init(&b[CB_D3_FULL], 1);
            mbar_init(&b[CB_D3_FREE], CH_EPI_WARPS);
        }
        mbar_init(w_full, 1);
        fence_barrier_init();
    }
    if (warp == CH_MMA_WARP) tmem_alloc<512>(tmem_holder);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    // tile j of slot s in iteration it: (it * gridDim.x + blockIdx.x) * CH_SLOTS + s
    auto tile_of = [&](int64_t it, int s) { return (it * (int64_t)gridDim.x + blockIdx.x) * CH_SLOTS + s; };

    if (warp >= CH_MMA_WARP && warp < CH_MMA_WARP + CH_SLOTS) {
        // ---------------------------------------------------------------- MMA issuer of slot s (whole warp, one elected lane)
        const int s = warp - CH_MMA_WARP;
        unsigned leader;
        asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(leader));
        if (s == 0 && leader) {   // the weight images, once
            const int total = p.w_bytes[0] + p.w_bytes[1] + p.w_bytes[2];
            mbar_expect_tx(w_full, (unsigned)total);
            for (int l = 0; l < 3; ++l) {
                uint8_t *dst = l == 0 ? W0 : (l == 1 ? W1 : W2);
                for (int off = 0; off < p.w_bytes[l]; off += 16384) bulk_g2s(dst + off, p.w_img[l] + off, 16384u, w_full);
            }
            mbar_arrive(w_full);
        }
        __syncwarp();
        mbar_wait(w_full, 0);
        const uint32_t idesc_k = idesc_16(128, CH_ROWS, false, false, FMT_F16, FMT_F16);   // layer 1: K-major B
        const uint32_t idesc_mn = idesc_16(128, CH_ROWS, false, true, FMT_F16, FMT_F16);   // layers 2, 3: MN-major B
        uint64_t *b = bars + s * CB_PER_SLOT;
        uint8_t *B1 = slots + s * slot_bytes;
        const uint64_t dw0 = smem_desc_sw128(smem_u32(W0), 16, ATOM_BYTES);
        const uint64_t dw1 = smem_desc_sw128(smem_u32(W1), 16, ATOM_BYTES);
        const uint64_t dw2 = smem_desc_sw128(smem_u32(W2), 16, ATOM_BYTES);
        const uint64_t db1 = smem_desc_sw128(smem_u32(B1), 16, ATOM_BYTES);                        // K-major gathered rows
        const uint64_t db2 = smem_desc_sw128(smem_u32(B1 + b1_bytes), 64 * LINE_BYTES, ATOM_BYTES);  // MN-major activations
        // descriptor address field is in 16-byte units: advancing an operand by `bytes` adds bytes >> 4
        constexpr uint64_t A_KS = 32 >> 4, A_CHUNK = (128 * LINE_BYTES) >> 4, B_KS_K = 32 >> 4,
                           B_KS_MN = (16 * LINE_BYTES) >> 4, B_CHUNK = CH_CHUNK_BYTES >> 4;
        const uint32_t d1 = tmem_base + s * CH_TMEM_PER_SLOT, d2 = d1 + 64, d3 = d1 + 128;
        for (int64_t it = 0;; ++it) {
            if (tile_of(it, s) >= num_tiles) break;
            const uint32_t ph = (uint32_t)(it & 1);
            // ---- layer 1
            mbar_wait(&b[CB_B1_FULL], ph);
            tc_fence_after();
            if (leader) {
#pragma unroll
                for (int kc = 0; kc < (K1C_ >= 0 ? K1C_ : 3); ++kc) {
                    if (kc < k1c) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks)
                            if (kc + 1 < k1c || ks < nks_last)
                                umma_bf16(d1, dw0 + kc * A_CHUNK + ks * A_KS, db1 + kc * B_CHUNK + ks * B_KS_K, idesc_k, (kc | ks) != 0);
                    }
                }
                umma_commit(&b[CB_B1_FREE]);
                umma_commit(&b[CB_D1_FULL]);
            }
            __syncwarp();
            // ---- layer 2
            mbar_wait(&b[CB_A1_FULL], ph);
            tc_fence_after();
            if (leader) {
#pragma unroll
                for (int kc = 0; kc < (C1C_ >= 0 ? C1C_ : 2); ++kc) {
                    if (kc < c1c) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks)
                            umma_bf16(d2, dw1 + kc * A_CHUNK + ks * A_KS, db2 + kc * B_CHUNK + ks * B_KS_MN, idesc_mn, (kc | ks) != 0);
                    }
                }
                umma_commit(&b[CB_D2_FULL]);
            }
            __syncwarp();
            // ---- layer 3 (its accumulator must have been drained by the previous tile's max)
            mbar_wait(&b[CB_A2_FULL], ph);
            mbar_wait(&b[CB_D3_FREE], ph ^ 1u);
            tc_fence_after();
            if (leader) {
#pragma unroll
                for (int mt = 0; mt < (MT3_ >= 0 ? MT3_ : 2); ++mt) {
                    if (mt < mt3) {
#pragma unroll
                        for (int kc = 0; kc < (C2C_ >= 0 ? C2C_ : 2); ++kc) {
                            if (kc < c2c) {
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks)
                                    umma_bf16(d3 + mt * 64, dw2 + (uint64_t)(kc * mt3 + mt) * A_CHUNK + ks * A_KS,
                                              db2 + kc * B_CHUNK + ks * B_KS_MN, idesc_mn, (kc | ks) != 0);
                            }
                        }
                    }
                }
                umma_commit(&b[CB_D3_FULL]);
            }
            __syncwarp();
        }
    } else if (warp >= CH_MMA_WARP + CH_SLOTS) {
        // ---------------------------------------------------------------- gather loaders: two threads per row of the tile
        const int lt0 = tid - (CH_MMA_WARP + CH_SLOTS) * 32;
        const int s = lt0 / CH_LOAD_THREADS, lt = lt0 % CH_LOAD_THREADS;
        const int r = lt >> 1, part = lt & 1;   // my row of the tile; my half of every 128-byte line (chunks 4 part .. 4 part + 3)
        uint64_t *b = bars + s * CB_PER_SLOT;
        uint8_t *B1 = slots + s * slot_bytes;
        // (source index, centroid) of my row in a tile: the head of the dependent chain, fetched one tile ahead
        auto fetch_idx = [&](int64_t tile, int &sidx, int &m) {
            sidx = -1;
            m = 0;
            const int64_t row = tile * CH_ROWS + r;
            if (tile < num_tiles && row < rows) {
                sidx = __ldg(gl.rm.row_src + row);
                m = gi_seg(__ldg(gl.rm.rgrp + (row >> 3)));
            }
        };
        int sidx, m;
        fetch_idx(tile_of(0, s), sidx, m);
        for (int64_t it = 0;; ++it) {
            const int64_t tile = tile_of(it, s);
            if (tile >= num_tiles) break;
            gl.set_row_idx(sidx, m);                  // position loads of my row
            uint4 v[3][4];                            // my chunks of the (at most three) K chunks
#pragma unroll
            for (int kc = 0; kc < 3; ++kc)
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    v[kc][c] = (kc < k1c && kc * KC + (part * 4 + c) * 8 < p.k_img) ? gl.chunk(kc * KC + (part * 4 + c) * 8)
                                                                         : make_uint4(0u, 0u, 0u, 0u);
            fetch_idx(tile_of(it + 1, s), sidx, m);   // next tile's indices: in flight while this tile is stored
            mbar_wait(&b[CB_B1_FREE], (uint32_t)(it & 1) ^ 1u);
#pragma unroll
            for (int kc = 0; kc < 3; ++kc) {
                if (kc < k1c) {
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        *reinterpret_cast<uint4 *>(B1 + kc * CH_CHUNK_BYTES + line_chunk_off(r, part * 4 + c)) = v[kc][c];
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&b[CB_B1_FULL]);
        }
    } else {
        // ---------------------------------------------------------------- epilogue group of slot s
        const int s = warp / CH_EPI_WARPS, w8 = warp % CH_EPI_WARPS;
        const int q = w8 & 3, half = w8 >> 2;
        uint64_t *b = bars + s * CB_PER_SLOT;
        uint8_t *X = slots + s * slot_bytes + b1_bytes;
        const int ch = q * 32 + lane;                                  // my channel within a 128-lane M tile
        const uint32_t lane_addr = ((uint32_t)(q * 32)) << 16;
        const uint32_t d1 = tmem_base + lane_addr + s * CH_TMEM_PER_SLOT, d2 = d1 + 64, d3 = d1 + 128;
        float sc1, sh1, sc2, sh2;
        chain_affine(p, 0, ch, sc1, sh1);
        chain_affine(p, 1, ch, sc2, sh2);
        const bool relu = p.act == B2PN_ACT_RELU;
        // layer 3: with two M tiles the column halves become M tiles (every thread scans all 64 rows of its channel)
        const int ch3 = (mt3 == 2 ? half * 128 : 0) + ch;
        const bool ep3 = mt3 == 2 || half == 0;
        const bool want_arg = p.arg != nullptr;
        const float b3 = (ep3 && ch3 < p.c3) ? p.bias[2][ch3] : 0.f;
        // my 32 rows of the tile as four 16-byte groups of my channel's line in the MN-major operand tile
        uint8_t *xline = X + (ch >> 6) * CH_CHUNK_BYTES + (ch & 63) * LINE_BYTES;
        const int sw = ch & 7;

        auto hidden = [&](uint32_t dcol, float sc, float sh, int C, uint64_t *full, uint64_t *ready, uint32_t ph) {
            mbar_wait(full, ph);
            tc_fence_after();
            if (ch - lane < C) {   // a warp whose 32 channels are all padding has nothing to drain
                float v[32];
                tmem_ld32(dcol + half * 32, v);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float f[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        float y = fmaf(v[8 * j + e], sc, sh);
                        f[e] = relu ? fmaxf(y, 0.f) : y;
                    }
                    *reinterpret_cast<uint4 *>(xline + (((half * 4 + j) ^ sw) << 4)) = pack8h(f);
                }
            }
            fence_proxy_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(ready);
        };

        for (int64_t it = 0;; ++it) {
            const int64_t tile = tile_of(it, s);
            if (tile >= num_tiles) break;
            const uint32_t ph = (uint32_t)(it & 1);
            // the tile's eight group descriptors (warp-uniform): requested now, needed after two more layers
            unsigned dsc[8];
#pragma unroll
            for (int g = 0; g < 8; ++g) {
                const int64_t gi = tile * (CH_ROWS / 8) + g;
                dsc[g] = (ep3 && gi * 8 < rows) ? __ldg(p.rgrp + gi) : GI_NONE;
            }
            hidden(d1, sc1, sh1, p.c1, &b[CB_D1_FULL], &b[CB_A1_FULL], ph);
            hidden(d2, sc2, sh2, p.c2, &b[CB_D2_FULL], &b[CB_A2_FULL], ph);
            // ---- layer 3 + max over the rows of every centroid of the tile
            mbar_wait(&b[CB_D3_FULL], ph);
            tc_fence_after();
            if (ep3 && ch3 - lane < p.c3) {
                const uint32_t dcol = d3 + (mt3 == 2 ? half * 64 : 0);
                float best = -INFINITY;
                int bk = -1;
#pragma unroll 1
                for (int cc = 0; cc < 2; ++cc) {
                    float v[32];
                    tmem_ld32(dcol + cc * 32, v);
#pragma unroll
                    for (int gg = 0; gg < 4; ++gg) {
                        const unsigned inf = cc == 0 ? dsc[gg] : dsc[4 + gg];  // warp-uniform
                        if (gi_none(inf)) continue;
                        const int s0 = gi_slot0(inf), nv = gi_nv(inf);
                        if (s0 == 0) {
                            best = -INFINITY;
                            bk = -1;
                        }
                        if (want_arg) {
#pragma unroll
                            for (int e = 0; e < 8; ++e) {
                                const float x = v[gg * 8 + e] + b3;
                                if (e < nv && x > best) {
                                    best = x;
                                    bk = s0 + e;
                                }
                            }
                        } else {   // evaluation: the value alone (bias added once per centroid below)
#pragma unroll
                            for (int e = 0; e < 8; ++e)
                                if (e < nv) best = fmaxf(best, v[gg * 8 + e]);
                            if (nv > 0) bk = 0;   // an empty neighbourhood (cnt = 0: one group, nv = 0) stays 0
                        }
                        if (gi_last(inf) && ch3 < p.c3) {
                            const int64_t m = gi_seg(inf);
                            const float o = bk >= 0 ? (want_arg ? best : best + b3) : 0.f;
                            p.out[m * p.c3 + ch3] = o;
                            if (want_arg) p.arg[m * p.c3 + ch3] = bk;
                            if (p.out16) p.out16[m * p.c3 + ch3] = __float2half_rn(o);
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&b[CB_D3_FREE]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == CH_MMA_WARP) tmem_dealloc<512>(tmem_base);
}

// =====================================================================================================================
//  Training passes.  Train-mode BatchNorm needs the batch statistics of a layer before its output can be normalised, so a
//  level cannot be one launch; but two consecutive layers CAN share one: the pass that normalises layer l also runs layer
//  l + 1 on the freshly normalised tile while it is still in shared memory.  The forward pass of a level becomes
//      A1  statistics of layer 1                                   (tc_rows_gemm_kernel<StatsEpTC>, sa_tc.cu)
//      P2  layer 1 -> normalise, store zhat1 / a1 -> layer 2 -> statistics of layer 2          (this kernel, PASS 2)
//      P3  a1 -> layer 2 -> normalise, store zhat2 / a2 -> layer 3 -> max + arg-max            (this kernel, PASS 3)
//  three GEMM passes instead of five, and a1 / a2 are read back once instead of twice (round-1 verdict: 31-38x the
//  compulsory bytes).  The input tile (g1 for P2, a1 for P3) is a stored feature-major tensor: one thread fetches it with
//  TMA tensor-map copies straight into the MN-major operand layout.
//
//   warps  0- 7 / 8-15   epilogue group of slot 0 / 1
//   warps 16 / 17        MMA issuer of slot 0 / 1 (whole warp, one elected lane; warp 16 owns the TMEM allocation)
//   warps 18 / 19        TMA producer of slot 0 / 1 (one elected lane)
// =====================================================================================================================
constexpr int CT_THREADS = CH_SLOTS * CH_EPI_THREADS + CH_SLOTS * 32 + CH_SLOTS * 32;  // 640
enum { TB_IN_FULL = 0, TB_IN_FREE, TB_DA_FULL, TB_XA_FULL, TB_DB_FULL, TB_DB_FREE, TB_PER_SLOT };

struct ChainTrainParams {
    const uint8_t *w_img[2];  // P2: layers 1, 2; P3: layers 2, 3 (fp16 images, num_mg == 1)
    int w_bytes[2];
    int k_in;                 // real K of the first GEMM (P2: image columns of g1; P3: c1)
    int kc_in, kc_mid;        // K chunks of the first / second GEMM
    int c_a, c_b;             // output channels of the first / second GEMM
    int mt_b;                 // M tiles of the second GEMM
    int64_t rows;
    const int64_t *rows_dev;
    int64_t ld;
    // first GEMM: zhat = (acc + bias - mean) * rstd; a = act(gamma * zhat + beta), invalid rows 0; both stored [c_a][ld]
    const float *bias_a, *mean_a, *rstd_a, *gamma_a, *beta_a;
    int dup_a;                // c_a == 64 and the first GEMM's image repeats its rows on lines 64..127 (PackJob::dup64)
    int act;
    __half *z_out, *a_out;
    // second GEMM: PASS 2 -> per-channel sum / sum of squares of the bias-free accumulators, per CTA and writer group:
    // partial[(blockIdx.x * 4 + slot * 2 + half)][2][cpad]; PASS 3 -> per-centroid max (+ bias) and arg-max slot
    double *partial;
    int cpad;
    const float *bias_b;
    float *out;
    int32_t *arg;
    __half *out16;
    const uint32_t *rgrp;
};

template <int PASS, int KCI_, int NKSL_, int KCM_, int MTB_>
__global__ void __launch_bounds__(CT_THREADS, 1)
    tc_chain_train_kernel(const ChainTrainParams p, const __grid_constant__ TmaMap map_in, const __grid_constant__ TmaMap map_z,
                          const __grid_constant__ TmaMap map_a)
{
    static_assert(PASS == 2 || PASS == 3, "PASS 2: layer 1 + statistics of layer 2; PASS 3: layer 2 + layer 3 + max");
    const int kc_in = KCI_ >= 0 ? KCI_ : p.kc_in;
    const int kc_mid = KCM_ >= 0 ? KCM_ : p.kc_mid;
    const int mt_b = MTB_ >= 0 ? MTB_ : p.mt_b;
    const int nks_last = NKSL_ >= 0 ? NKSL_ : ((p.k_in - (p.kc_in - 1) * KC) >= KC ? 4 : (p.k_in - (p.kc_in - 1) * KC + 15) / 16);
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t *Wa = smem, *Wb = Wa + p.w_bytes[0];
    uint8_t *slots = Wb + p.w_bytes[1];
    // per slot: IN (the fetched input tile), X (a: operand of the second GEMM AND source of its TMA store), Z (zhat staging)
    const int in_bytes = kc_in * CH_CHUNK_BYTES, x_bytes = kc_mid * CH_CHUNK_BYTES;
    const int slot_bytes = in_bytes + 2 * x_bytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(slots + CH_SLOTS * slot_bytes);
    uint64_t *w_full = bars + CH_SLOTS * TB_PER_SLOT;
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(w_full + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t rows = p.rows_dev ? *p.rows_dev : p.rows;
    // whole 128-row tiles, like every other consumer of the stored tensors: the pad rows of the last one get a = 0
    const int64_t num_tiles = ((rows + 127) / 128) * 2;

    if (tid == 0) {
        for (int s = 0; s < CH_SLOTS; ++s) {
            uint64_t *b = bars + s * TB_PER_SLOT;
            mbar_init(&b[TB_IN_FULL], 1);
            mbar_init(&b[TB_IN_FREE], 1);
            mbar_init(&b[TB_DA_FULL], 1);
            mbar_init(&b[TB_XA_FULL], 1);
            mbar_init(&b[TB_DB_FULL], 1);
            mbar_init(&b[TB_DB_FREE], CH_EPI_WARPS);
        }
        mbar_init(w_full, 1);
        fence_barrier_init();
    }
    if (warp == CH_MMA_WARP) tmem_alloc<512>(tmem_holder);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    auto tile_of = [&](int64_t it, int s) { return (it * (int64_t)gridDim.x + blockIdx.x) * CH_SLOTS + s; };
    unsigned leader;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(leader));

    if (warp >= CH_MMA_WARP + CH_SLOTS) {
        // ---------------------------------------------------------------- TMA producer of slot s
        const int s = warp - (CH_MMA_WARP + CH_SLOTS);
        if (s < CH_SLOTS && leader) {
            uint64_t *b = bars + s * TB_PER_SLOT;
            uint8_t *IN = slots + s * slot_bytes;
            for (int64_t it = 0;; ++it) {
                const int64_t tile = tile_of(it, s);
                if (tile >= num_tiles) break;
                mbar_wait(&b[TB_IN_FREE], (uint32_t)(it & 1) ^ 1u);
                mbar_expect_tx(&b[TB_IN_FULL], (unsigned)in_bytes);
                for (int kc = 0; kc < kc_in; ++kc)
                    tma_load_2d(IN + kc * CH_CHUNK_BYTES, &map_in, (int)(tile * CH_ROWS), kc * KC, &b[TB_IN_FULL]);
                mbar_arrive(&b[TB_IN_FULL]);
            }
        }
    } else if (warp >= CH_MMA_WARP) {
        // ---------------------------------------------------------------- MMA issuer of slot s
        const int s = warp - CH_MMA_WARP;
        if (s == 0 && leader) {
            mbar_expect_tx(w_full, (unsigned)(p.w_bytes[0] + p.w_bytes[1]));
            for (int l = 0; l < 2; ++l) {
                uint8_t *dst = l == 0 ? Wa : Wb;
                for (int off = 0; off < p.w_bytes[l]; off += 16384) bulk_g2s(dst + off, p.w_img[l] + off, 16384u, w_full);
            }
            mbar_arrive(w_full);
        }
        __syncwarp();
        mbar_wait(w_full, 0);
        const uint32_t idesc_mn = idesc_16(128, CH_ROWS, false, true, FMT_F16, FMT_F16);
        uint64_t *b = bars + s * TB_PER_SLOT;
        uint8_t *IN = slots + s * slot_bytes;
        const uint64_t dwa = smem_desc_sw128(smem_u32(Wa), 16, ATOM_BYTES);
        const uint64_t dwb = smem_desc_sw128(smem_u32(Wb), 16, ATOM_BYTES);
        const uint64_t din = smem_desc_sw128(smem_u32(IN), 64 * LINE_BYTES, ATOM_BYTES);
        const uint64_t dx = smem_desc_sw128(smem_u32(IN + in_bytes), 64 * LINE_BYTES, ATOM_BYTES);
        constexpr uint64_t A_KS = 32 >> 4, A_CHUNK = (128 * LINE_BYTES) >> 4, B_KS_MN = (16 * LINE_BYTES) >> 4,
                           B_CHUNK = CH_CHUNK_BYTES >> 4;
        const uint32_t da = tmem_base + s * CH_TMEM_PER_SLOT, db = da + 64;
        for (int64_t it = 0;; ++it) {
            if (tile_of(it, s) >= num_tiles) break;
            const uint32_t ph = (uint32_t)(it & 1);
            mbar_wait(&b[TB_IN_FULL], ph);
            tc_fence_after();
            if (leader) {
#pragma unroll
                for (int kc = 0; kc < (KCI_ >= 0 ? KCI_ : 3); ++kc) {
                    if (kc < kc_in) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks)
                            if (kc + 1 < kc_in || ks < nks_last)
                                umma_bf16(da, dwa + kc * A_CHUNK + ks * A_KS, din + kc * B_CHUNK + ks * B_KS_MN, idesc_mn, (kc | ks) != 0);
                    }
                }
                umma_commit(&b[TB_IN_FREE]);
                umma_commit(&b[TB_DA_FULL]);
            }
            __syncwarp();
            mbar_wait(&b[TB_XA_FULL], ph);
            mbar_wait(&b[TB_DB_FREE], ph ^ 1u);
            tc_fence_after();
            if (leader) {
#pragma unroll
                for (int mt = 0; mt < (MTB_ >= 0 ? MTB_ : 2); ++mt) {
                    if (mt < mt_b) {
#pragma unroll
                        for (int kc = 0; kc < (KCM_ >= 0 ? KCM_ : 2); ++kc) {
                            if (kc < kc_mid) {
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks)
                                    umma_bf16(db + mt * 64, dwb + (uint64_t)(kc * mt_b + mt) * A_CHUNK + ks * A_KS,
                                              dx + kc * B_CHUNK + ks * B_KS_MN, idesc_mn, (kc | ks) != 0);
                            }
                        }
                    }
                }
                umma_commit(&b[TB_DB_FULL]);
            }
            __syncwarp();
        }
    } else {
        // ---------------------------------------------------------------- epilogue group of slot s
        const int s = warp / CH_EPI_WARPS, w8 = warp % CH_EPI_WARPS;
        const int q = w8 & 3, half = w8 >> 2;
        uint64_t *b = bars + s * TB_PER_SLOT;
        uint8_t *X = slots + s * slot_bytes + in_bytes;
        const int ch = q * 32 + lane;
        const uint32_t lane_addr = ((uint32_t)(q * 32)) << 16;
        const uint32_t da = tmem_base + lane_addr + s * CH_TMEM_PER_SLOT, db = da + 64;
        // first GEMM with 64 output channels: the weight image repeats its rows (PackJob::dup64), channel c sits on TMEM lanes
        // c and 64 + c, and the eight warps split the tile as (32-channel half, 16-column quarter) instead of leaving the
        // warps of lane quadrants 2 and 3 idle while the other four drain 32 columns each
        const bool dup = (KCM_ == 1 || KCM_ < 0) && p.dup_a != 0;   // 64 channels <=> one K chunk of the second GEMM
        const int cha = dup ? (q & 1) * 32 + lane : ch;            // my channel of the first GEMM
        const int col16 = half * 2 + (q >> 1);                      // dup: my 16-column quarter
        float sc = 0.f, sh = 0.f, ga = 0.f, be = 0.f;
        if (cha < p.c_a) {
            sc = p.rstd_a[cha];
            sh = (p.bias_a[cha] - p.mean_a[cha]) * sc;
            ga = p.gamma_a[cha];
            be = p.beta_a[cha];
        }
        const bool relu = p.act == B2PN_ACT_RELU;
        const int chb = (PASS == 3 && mt_b == 2 ? half * 128 : 0) + ch;   // my channel of the second GEMM
        const bool epb = PASS == 2 || mt_b == 2 || half == 0;
        const float bb = (PASS == 3 && epb && chb < p.c_b) ? p.bias_b[chb] : 0.f;
        uint8_t *xline = X + (cha >> 6) * CH_CHUNK_BYTES + (cha & 63) * LINE_BYTES;
        const int sw = cha & 7;
        double S = 0.0, Q = 0.0;   // PASS 2: statistics of my channel over all my tiles
        // the eight group descriptors of a tile (warp-uniform, 32 contiguous bytes of the table) are requested one tile
        // ahead as RAW words: the load used to sit at the top of the tile and the whole group waited an L2 round trip for it
        // (16 % of the epilogue warps' samples, ncu round 2).  The table is allocated in whole tiles, so the read is in bounds.
        uint4 nx0 = make_uint4(GI_NONE, GI_NONE, GI_NONE, GI_NONE), nx1 = nx0;
        if (tile_of(0, s) < num_tiles) {
            const uint4 *t = reinterpret_cast<const uint4 *>(p.rgrp + tile_of(0, s) * (CH_ROWS / 8));
            nx0 = __ldg(t);
            nx1 = __ldg(t + 1);
        }
        for (int64_t it = 0;; ++it) {
            const int64_t tile = tile_of(it, s);
            if (tile >= num_tiles) break;
            const uint32_t ph = (uint32_t)(it & 1);
            const int64_t row0 = tile * CH_ROWS;
            unsigned dsc[8] = {nx0.x, nx0.y, nx0.z, nx0.w, nx1.x, nx1.y, nx1.z, nx1.w};
#pragma unroll
            for (int g = 0; g < 8; ++g) {
                const int64_t gi = tile * (CH_ROWS / 8) + g;
                if (gi * 8 >= rows || gi_none(dsc[g])) dsc[g] = GI_NONE;
            }
            if (tile_of(it + 1, s) < num_tiles) {
                const uint4 *t = reinterpret_cast<const uint4 *>(p.rgrp + tile_of(it + 1, s) * (CH_ROWS / 8));
                nx0 = __ldg(t);
                nx1 = __ldg(t + 1);
            }
            // ---- first GEMM: normalise; zhat and a leave through shared-memory tiles and TMA stores (16-byte global stores
            // 2*ld bytes apart per lane made this epilogue 3x slower, as they had in round 1); a is also the operand of
            // the second GEMM, read in place
            mbar_wait(&b[TB_DA_FULL], ph);
            tc_fence_after();
            if (w8 == 0 && lane == 0) bulk_wait_read_all();      // the previous tile's stores have read X and Z
            asm volatile("bar.sync %0, %1;" ::"r"(1 + s), "n"(CH_EPI_THREADS) : "memory");
            if (dup) {
                unsigned nv2 = 0u;   // valid rows of my two 8-row groups
#pragma unroll
                for (int g = 0; g < 8; ++g)
                    if ((g >> 1) == col16) nv2 |= (unsigned)gi_nv(dsc[g]) << (4 * (g & 1));
                float v[16];
                tmem_ld16(da + col16 * 16, v);
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int nv = (int)((nv2 >> (4 * j)) & 15u);
                    float f[8], g[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) f[e] = fmaf(v[8 * j + e], sc, sh);
                    const uint4 zq = pack8h(f);
                    unpack8h(zq, f);
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        float y = fmaf(f[e], ga, be);
                        if (relu) y = fmaxf(y, 0.f);
                        g[e] = e < nv ? y : 0.f;
                    }
                    const int off = ((col16 * 2 + j) ^ sw) << 4;
                    *reinterpret_cast<uint4 *>(xline + x_bytes + off) = zq;
                    *reinterpret_cast<uint4 *>(xline + off) = pack8h(g);
                }
            } else if (ch - lane < p.c_a) {
                float v[32];
                tmem_ld32(da + half * 32, v);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int nv = gi_nv(half == 0 ? dsc[j] : dsc[4 + j]);
                    float f[8], g[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) f[e] = fmaf(v[8 * j + e], sc, sh);
                    const uint4 zq = pack8h(f);
                    unpack8h(zq, f);   // the activation is defined on the STORED (fp16) zhat, as backward recomputes it
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        float y = fmaf(f[e], ga, be);
                        if (relu) y = fmaxf(y, 0.f);
                        g[e] = e < nv ? y : 0.f;
                    }
                    const int off = ((half * 4 + j) ^ sw) << 4;
                    *reinterpret_cast<uint4 *>(xline + x_bytes + off) = zq;        // Z tile (behind X)
                    *reinterpret_cast<uint4 *>(xline + off) = pack8h(g);           // X tile
                }
            }
            fence_proxy_async_smem();
            tc_fence_before();
            asm volatile("bar.sync %0, %1;" ::"r"(1 + s), "n"(CH_EPI_THREADS) : "memory");
            if (w8 == 0 && lane == 0) {
                for (int kc = 0; kc < kc_mid; ++kc) {   // channels past c_a are clipped by the tensor maps
                    tma_store_2d(&map_z, X + x_bytes + kc * CH_CHUNK_BYTES, (int)row0, kc * KC);
                    tma_store_2d(&map_a, X + kc * CH_CHUNK_BYTES, (int)row0, kc * KC);
                }
                bulk_commit_group();
                mbar_arrive(&b[TB_XA_FULL]);
            }
            // ---- second GEMM
            mbar_wait(&b[TB_DB_FULL], ph);
            tc_fence_after();
            if (PASS == 2) {
                if (ch - lane < p.c_b) {
                    float v[32];
                    tmem_ld32(db + half * 32, v);
                    float sm = 0.f, qm = 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        sm += v[j];
                        qm = fmaf(v[j], v[j], qm);
                    }
                    S += (double)sm;
                    Q += (double)qm;
                }
            } else if (epb && chb - lane < p.c_b) {
                const uint32_t dcol = db + (mt_b == 2 ? half * 64 : 0);
                float best = -INFINITY;
                int bk = -1;
#pragma unroll 1
                for (int cc = 0; cc < 2; ++cc) {
                    float v[32];
                    tmem_ld32(dcol + cc * 32, v);
#pragma unroll
                    for (int gg = 0; gg < 4; ++gg) {
                        const unsigned inf = cc == 0 ? dsc[gg] : dsc[4 + gg];
                        if (gi_none(inf)) continue;
                        const int s0 = gi_slot0(inf), nv = gi_nv(inf);
                        if (s0 == 0) {
                            best = -INFINITY;
                            bk = -1;
                        }
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const float x = v[gg * 8 + e] + bb;
                            if (e < nv && x > best) {
                                best = x;
                                bk = s0 + e;
                            }
                        }
                        if (gi_last(inf) && chb < p.c_b) {
                            const int64_t m = gi_seg(inf);
                            const float o = bk >= 0 ? best : 0.f;
                            p.out[m * p.c_b + chb] = o;
                            p.arg[m * p.c_b + chb] = bk;
                            if (p.out16) p.out16[m * p.c_b + chb] = __float2half_rn(o);
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&b[TB_DB_FREE]);
        }
        if (w8 == 0 && lane == 0) bulk_wait_all();
        if (PASS == 2 && ch < p.c_b) {   // every (CTA, writer group) writes its slice, tiles or not: the finalize sums them all
            double *pt = p.partial + ((int64_t)blockIdx.x * 4 + s * 2 + half) * 2 * p.cpad;
            pt[ch] = S;
            pt[p.cpad + ch] = Q;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == CH_MMA_WARP) tmem_dealloc<512>(tmem_base);
}

static int chain_train_smem_bytes(const ChainTrainParams &p)
{
    return p.w_bytes[0] + p.w_bytes[1] + CH_SLOTS * (p.kc_in + 2 * p.kc_mid) * CH_CHUNK_BYTES + 256 + 1024;
}

// SLOTS levels whose shapes the chained kernels cover (the reference's levels 1 and 2 with neuron_multiplier 1): hidden
// widths of whole 64-channel chunks up to 128, output up to 256 channels, and at most three 64-column chunks of the
// layer-1 operand, `k_lines` of which the kernel reads.  The callers add the mode: evaluation with h1 == NULL
// (tc_chain_eval_kernel), or training with g1 materialised (tc_chain_train_kernel)
static bool chain_shapes_ok(const b2pn_sa_args &a, int k_lines, int c1, int c2, int c3)
{
    return a.seg_mode == B2PN_SEG_SLOTS && c1 % 64 == 0 && c2 % 64 == 0 && c1 <= 128 && c2 <= 128 && c3 <= 256 &&
           k_lines <= 3 * KC;
}

static int chain_smem_bytes(const ChainParams &p)
{
    const int x_bytes = (p.c1c > p.c2c ? p.c1c : p.c2c) * CH_CHUNK_BYTES;
    return p.w_bytes[0] + p.w_bytes[1] + p.w_bytes[2] + CH_SLOTS * (p.k1c * CH_CHUNK_BYTES + x_bytes) + 256 + 1024;
}

}  // namespace tc
}  // namespace b2pn
