// Kernel 3, bf16 mode -- set-abstraction MLP on the 5th-generation tensor cores (tcgen05 + TMEM).
//
// Orientation: every layer computes the TRANSPOSED product  D^T[channel, row] = W[channel, k] * A^T[k, row]
// so that output channels sit on the 128 TMEM lanes and rows (neighbour slots / points) on the TMEM
// columns.  One epilogue thread then owns one channel: BatchNorm statistics are two registers per
// thread, the per-centroid max over its K slots is a per-thread scan of K consecutive accumulator
// columns (no shuffles, no atomics), and activations are stored FEATURE-MAJOR (hT[channel][row]) with
// 16-byte vector stores.  Feature-major activations are exactly the MN-major B operand of the next
// layer and the K-major operands of the dW GEMMs, so no transposes are ever needed.
//
// Pipeline of the rows kernel (persistent CTAs): a producer thread fetches the B tile with two TMA tensor-map copies of a
// stored feature-major tensor (or, for the few operands that still need arithmetic on the way in, two groups of SIMT
// loader warps build it) and the pre-packed weight chunk with a bulk copy; one thread issues tcgen05.mma; the epilogue
// warps -- two groups of eight when the operands come by TMA, one group per TMEM accumulator buffer -- drain TMEM and
// send result tiles out through shared-memory staging tiles and TMA stores.  K is streamed in chunks of 64 through a
// ring of shared-memory stages.  tc_dw_kernel is the same machinery with K = rows and the accumulator kept in TMEM
// over the CTA's whole row range.
#include <cuda.h>  // CUtensorMap types only; the encoder is fetched through the runtime (no libcuda link)
#include <math.h>

#include "tc_common.cuh"

namespace b2pn {
namespace tc {

constexpr int R = 128;          // rows per tile = UMMA N
constexpr int KC = 64;          // reduction chunk = one 128-byte line of bf16
constexpr int NUM_EPI = 256;    // warps 0-7: warp w drains TMEM lanes 32*(w%4).., column half w/4
constexpr int NUM_LOAD = 128;   // threads per loader group
constexpr int LOAD_GROUPS = 2;  // warps 8-11 and 12-15 fill alternate pipeline stages (hides global-load latency)
constexpr int MMA_WARP = (NUM_EPI + LOAD_GROUPS * NUM_LOAD) / 32;  // warp 16: MMA issuer / TMEM owner
constexpr int NT = NUM_EPI + LOAD_GROUPS * NUM_LOAD + 32;
// TMA-fed rows kernels need no loader warps: warps 8-15 become a SECOND epilogue group (group g drains the tiles of
// parity g, i.e. TMEM accumulator buffer g), warp 16 issues the MMAs and warp 17 the TMA copies
constexpr int NT_TMA = 2 * NUM_EPI + 64;
constexpr int PROD_WARP_TMA = MMA_WARP + 1;
// wide layout with SIMT loaders: warps 0-15 two epilogue groups, warp 16 MMA, warps 17-20 one loader group
constexpr int NT_WIDE = 2 * NUM_EPI + 32 + NUM_LOAD;
constexpr int B_BYTES = R * LINE_BYTES;  // 16 KB: [128 row lines x 64 k] or [2 row blocks][64 k lines x 64 rows]

// Row structure of a level.
//   CLOUDS: row = source point, all rows < rows are valid.
//   SLOTS:  rows are the COMPACTED neighbour slots built by b2pn_pack_rows (pack_rows.cu): per 8-row group one
//           descriptor word (centroid, first slot, valid rows, last-group flag), per row the gathered source index.
//           The number of rows is only known on the device (rows_dev); kernels call resolve() first.
constexpr unsigned GI_NONE = 0x00ffffffu;  // no centroid, 0 valid rows
__device__ __forceinline__ int gi_seg(unsigned b) { return (int)(b & 0xffffffu); }
__device__ __forceinline__ bool gi_none(unsigned b) { return (b & 0xffffffu) == 0xffffffu; }
__device__ __forceinline__ int gi_slot0(unsigned b) { return (int)((b >> 24) & 7u) << 3; }
__device__ __forceinline__ int gi_nv(unsigned b) { return (int)((b >> 27) & 15u); }
__device__ __forceinline__ bool gi_last(unsigned b) { return (b >> 31) != 0u; }

struct RowMapTC {
    int seg_mode;
    const uint32_t *rgrp;     // SLOTS: [rows/8] group descriptors
    const int32_t *row_src;   // SLOTS: [rows] source point of the row, -1 = padding
    const int32_t *cnt;       // SLOTS: [n_dst]
    const int64_t *batch;     // CLOUDS: [rows] sorted cloud id
    int64_t rows;             // logical rows; SLOTS: filled in on the device (resolve) from b2pn_pack_rows' scalar
    int64_t n_dst;
    __device__ __forceinline__ void resolve(int64_t r) { rows = r; }
    // descriptor of the 8 rows starting at r8 (r8 % 8 == 0), normalised: nv == 0 wherever nothing is valid
    __device__ __forceinline__ unsigned info(int64_t r8) const
    {
        if (r8 >= rows) return GI_NONE;
        if (seg_mode) return GI_NONE | ((unsigned)min((int64_t)8, rows - r8) << 27);
        const unsigned b = __ldg(rgrp + (r8 >> 3));
        return gi_none(b) ? GI_NONE : b;
    }
    __device__ __forceinline__ int valid8(int64_t r8) const { return gi_nv(info(r8)); }
    // valid rows (0..8) of the eight 8-row groups of the 64 rows starting at row0 (row0 % 64 == 0, below the row
    // capacity), packed 4 bits per group: two 16-byte descriptor loads and no branch (SLOTS), or arithmetic (CLOUDS)
    __device__ __forceinline__ unsigned valid64(int64_t row0) const
    {
        const int64_t left64 = rows - row0;
        const int left = left64 > 64 ? 64 : (left64 < 0 ? 0 : (int)left64);  // logical rows among my 64
        unsigned out = 0u;
        if (seg_mode) {
#pragma unroll
            for (int g = 0; g < 8; ++g) out |= (unsigned)min(max(left - 8 * g, 0), 8) << (4 * g);
            return out;
        }
        const uint4 *p = reinterpret_cast<const uint4 *>(rgrp + (row0 >> 3));
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        const unsigned d[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            const bool dead = 8 * g >= left || gi_none(d[g]);
            out |= (dead ? 0u : (unsigned)gi_nv(d[g])) << (4 * g);
        }
        return out;
    }
    // SLOTS only, r8 below the row capacity: the same word without a branch around the load, so that a loader
    // thread's eight descriptor loads (and what depends on them) go out back to back
    __device__ __forceinline__ unsigned info_slots(int64_t r8) const
    {
        const unsigned b = __ldg(rgrp + (r8 >> 3));
        return (r8 >= rows || gi_none(b)) ? GI_NONE : b;
    }
};

// ---- TMA tensor maps ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}
// box = 64 rows (128 bytes, the swizzle span) x 64 channels; channels past `channels` read as zeros
int make_tma_feature_major(TmaMap *out, const void *base, int64_t channels, int64_t ld, int box_channels)
{
    static_assert(sizeof(CUtensorMap) == sizeof(TmaMap), "CUtensorMap is 128 bytes");
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return B2PN_ENOTSUP;
    if (!base || channels <= 0 || ld <= 0 || (ld & 7) || ((uintptr_t)base & 15u)) return B2PN_EINVAL;
    const cuuint64_t dims[2] = {(cuuint64_t)ld, (cuuint64_t)channels};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 2u};
    const cuuint32_t box[2] = {64u, (cuuint32_t)box_channels};
    const cuuint32_t estr[2] = {1u, 1u};
    const CUresult r = fn(reinterpret_cast<CUtensorMap *>(out), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims,
                          strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? B2PN_OK : B2PN_EINVAL;
}

// the row-valid vector as a [1][ld] tensor: a 64-row x 16-line box whose first line is the vector, the rest zeros
int make_tma_row_valid(TmaMap *out, const void *base, int64_t ld)
{
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return B2PN_ENOTSUP;
    if (!base || ld <= 0 || (ld & 7) || ((uintptr_t)base & 15u)) return B2PN_EINVAL;
    const cuuint64_t dims[2] = {(cuuint64_t)ld, 1u};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 2u};
    const cuuint32_t box[2] = {64u, 16u};
    const cuuint32_t estr[2] = {1u, 1u};
    const CUresult r = fn(reinterpret_cast<CUtensorMap *>(out), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims,
                          strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? B2PN_OK : B2PN_EINVAL;
}

struct GemmParams {
    const uint8_t *a_packed;  // [m_group][k_chunk][MT*128 lines][128 B], swizzled 16-bit (a_fmt)
    int a_fmt, b_fmt;         // FMT_F16 / FMT_BF16 of the weight image and of the B operand tiles
    int num_kc;
    int64_t rows;             // host value (CLOUDS, self-test) ...
    const int64_t *rows_dev;  // ... or the device scalar of the compacted SLOTS layout (wins when non-NULL)
};

// layer-1 operand columns: [x (c_in) | x_lo (c_in, only when x arrives in fp32) | dpos_hi (3) | dpos_lo (3)].
// Raw fp32 inputs (intensity, relative positions) are split into bf16 hi + lo parts that meet the SAME
// weight column, so the tensor cores see them with ~16 mantissa bits at no extra MMA cost (the columns
// live in the padding of the 64-wide K chunk).
struct InCols {
    int c_in;
    int x_f32;
    __host__ __device__ int nx() const { return c_in * (x_f32 ? 2 : 1); }
    __host__ __device__ int k_img() const { return nx() + 6; }
    __host__ __device__ int src_col(int k) const  // weight column that feeds image column k (-1: padding)
    {
        const int n = nx();
        if (k < n) return k < c_in ? k : k - c_in;
        const int j = k - n;
        if (j < 3) return c_in + j;
        if (j < 6) return c_in + j - 3;
        return -1;
    }
};

__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16(v)); }
// forward-domain values are fp16 (tc_common.cuh): the hi part of an fp32 input and what is left of it
__device__ __forceinline__ float f16_round(float v) { return __half2float(__float2half_rn(v)); }

// fp16 twins (forward-domain tensors: zhat, activation operands, level outputs handed to the next level)
__device__ __forceinline__ void unpack8h(const uint4 &raw, float (&f)[8])
{
    const float2 a = unpack_f16x2(raw.x), b = unpack_f16x2(raw.y), c = unpack_f16x2(raw.z), d = unpack_f16x2(raw.w);
    f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ uint4 pack8h(const float (&f)[8])
{
    uint4 o;
    o.x = pack_f16x2(f[0], f[1]);
    o.y = pack_f16x2(f[2], f[3]);
    o.z = pack_f16x2(f[4], f[5]);
    o.w = pack_f16x2(f[6], f[7]);
    return o;
}
__device__ __forceinline__ void unpack8(const uint4 &raw, float (&f)[8])
{
    f[0] = bf16_lo(raw.x); f[1] = bf16_hi(raw.x); f[2] = bf16_lo(raw.y); f[3] = bf16_hi(raw.y);
    f[4] = bf16_lo(raw.z); f[5] = bf16_hi(raw.z); f[6] = bf16_lo(raw.w); f[7] = bf16_hi(raw.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8])
{
    uint4 o;
    o.x = pack_bf16x2(f[0], f[1]);
    o.y = pack_bf16x2(f[2], f[3]);
    o.z = pack_bf16x2(f[4], f[5]);
    o.w = pack_bf16x2(f[6], f[7]);
    return o;
}

// eight fp16 values -> eight bf16 values (exact range, 10 -> 7 mantissa bits): stored activations meeting bf16 gradients
__device__ __forceinline__ uint4 f16_to_bf16_chunk(const uint4 &raw)
{
    float f[8];
    unpack8h(raw, f);
    return pack8(f);
}

// =================================================================================================
//  B-tile loaders for the rows GEMM (128 threads).  produce() fills one 16 KB chunk for K chunk kc.
// =================================================================================================
struct GatherLoaderTC {  // K-major B: line = row of the tile, 64 k per line
    static constexpr bool B_MN = false;
    static constexpr bool USES_TMA = false;
    static constexpr bool WIDE = false;
    RowMapTC rm;
    const void *x;  // [n_src, c_in] row-major, fp32 (cols.x_f32) or fp16
    InCols cols;
    const float *pos_src;
    const float *pos_dst;
    int ones_col;  // image column that carries 1 for valid rows (dW bias column), -1: none
    int out_fmt;   // FMT_F16: forward operand / materialised g1; FMT_BF16: X side of a dW GEMM (meets bf16 gradients)
    // per-thread state for the current row
    bool ok;
    int64_t src;
    float d0, d1, d2;
    __device__ __forceinline__ void resolve(int64_t r) { rm.resolve(r); }
    __device__ __forceinline__ void set_row(int64_t row)
    {
        ok = row < rm.rows;
        src = 0;
        d0 = d1 = d2 = 0.f;
        if (ok && !rm.seg_mode) {
            const int sidx = __ldg(rm.row_src + row);
            ok = sidx >= 0;
            src = ok ? sidx : 0;
        } else if (ok) {
            src = row;
        }
        if (ok) {
            d0 = pos_src[3 * src + 0];
            d1 = pos_src[3 * src + 1];
            d2 = pos_src[3 * src + 2];
            if (!rm.seg_mode) {
                const int64_t m = gi_seg(__ldg(rm.rgrp + (row >> 3)));
                d0 = __fsub_rn(d0, pos_dst[3 * m + 0]);
                d1 = __fsub_rn(d1, pos_dst[3 * m + 1]);
                d2 = __fsub_rn(d2, pos_dst[3 * m + 2]);
            }
        }
    }
    // SLOTS rows whose (source index, centroid) the caller has already fetched (sidx < 0: padding row)
    __device__ __forceinline__ void set_row_idx(int sidx, int m)
    {
        ok = sidx >= 0;
        src = ok ? sidx : 0;
        d0 = d1 = d2 = 0.f;
        if (ok) {
            d0 = __fsub_rn(__ldg(pos_src + 3 * src + 0), __ldg(pos_dst + 3 * (int64_t)m + 0));
            d1 = __fsub_rn(__ldg(pos_src + 3 * src + 1), __ldg(pos_dst + 3 * (int64_t)m + 1));
            d2 = __fsub_rn(__ldg(pos_src + 3 * src + 2), __ldg(pos_dst + 3 * (int64_t)m + 2));
        }
    }
    __device__ __forceinline__ void begin_tile(int64_t tile, int lt) { set_row(tile * R + lt); }
    __device__ __forceinline__ float elem(int k) const
    {
        if (k == ones_col) return 1.f;
        const int c_in = cols.c_in, nx = cols.nx();
        if (k < c_in) {
            return cols.x_f32 ? reinterpret_cast<const float *>(x)[src * c_in + k]
                              : __half2float(reinterpret_cast<const __half *>(x)[src * c_in + k]);
        }
        if (k < nx) {
            const float v = reinterpret_cast<const float *>(x)[src * c_in + (k - c_in)];
            return v - (out_fmt == FMT_F16 ? f16_round(v) : bf16_round(v));
        }
        const int j = k - nx;
        if (j >= 6) return 0.f;
        const int a = j < 3 ? j : j - 3;
        const float v = a == 0 ? d0 : (a == 1 ? d1 : d2);
        return j < 3 ? v : v - (out_fmt == FMT_F16 ? f16_round(v) : bf16_round(v));
    }
    // 16-byte chunk holding image columns kk .. kk+7 of the current row
    __device__ __forceinline__ uint4 chunk(int kk) const
    {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (!ok) return v;
        if (!cols.x_f32 && (cols.c_in & 7) == 0 && kk + 8 <= cols.c_in) {
            v = __ldg(reinterpret_cast<const uint4 *>(reinterpret_cast<const __half *>(x) + src * cols.c_in + kk));
            return out_fmt == FMT_F16 ? v : f16_to_bf16_chunk(v);
        }
        if (kk < cols.k_img() + (ones_col >= 0 ? 1 : 0)) {
            float f[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = elem(kk + e);
            v = out_fmt == FMT_F16 ? pack8h(f) : pack8(f);
        }
        return v;
    }
    __device__ __forceinline__ void produce(uint8_t *B, int kc, int lt) const
    {
#pragma unroll
        for (int c = 0; c < 8; ++c) *reinterpret_cast<uint4 *>(B + line_chunk_off(lt, c)) = chunk(kc * KC + c * 8);
    }
    static __device__ __forceinline__ uint64_t b_desc(uint32_t b_saddr, int ks) { return smem_desc_sw128(b_saddr + ks * 32, 16, ATOM_BYTES); }
};

// Layer-1 operand materialised once: G[k][row] (bf16, feature-major) = image column k of the gathered + concatenated
// row ([x | x_lo | dpos_hi | dpos_lo | 1]), so that the statistics pass, the normalising pass and the dW1 GEMM all
// read it through TMA instead of gathering three times in their loader warps.  A block transposes 64 rows through
// shared memory: rows are gathered with 16-byte loads where the features allow it, columns leave as 128-byte lines.
constexpr int GATHER_ROWS = 64;
__global__ void __launch_bounds__(256) gather_l1_tc_kernel(GatherLoaderTC gl, const int64_t *rows_dev, int kg, int64_t ld,
                                                          __nv_bfloat16 *G)
{
    extern __shared__ __align__(16) unsigned char gth_smem[];
    __nv_bfloat16 *S = reinterpret_cast<__nv_bfloat16 *>(gth_smem);  // [kg8][64 rows]
    const int64_t rows = rows_dev ? *rows_dev : gl.rm.rows;
    gl.resolve(rows);
    const int64_t r0 = (int64_t)blockIdx.x * GATHER_ROWS;
    if (r0 >= (rows + 127) / 128 * 128) return;  // whole tiles, like every consumer
    const int kg8 = (kg + 7) & ~7;
    const int rl = threadIdx.x & 63, q = threadIdx.x >> 6;  // my row of the block, my chunk phase (0..3)
    gl.set_row(r0 + rl);
    for (int kk = q * 8; kk < kg8; kk += 32) {
        const uint4 v = gl.chunk(kk);
        const __nv_bfloat16 *e = reinterpret_cast<const __nv_bfloat16 *>(&v);
#pragma unroll
        for (int j = 0; j < 8; ++j) S[(kk + j) * GATHER_ROWS + rl] = e[j];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kg8 * 8; i += 256) {  // 8 chunks of 16 bytes per column line
        const int k = i >> 3, part = i & 7;
        if (k < kg)
            *reinterpret_cast<uint4 *>(G + (int64_t)k * ld + r0 + part * 8) =
                *reinterpret_cast<const uint4 *>(S + k * GATHER_ROWS + part * 8);
    }
}

// 8 consecutive rows (r8 .. r8+7) of channel ch of a feature-major tensor, as the B/A operand wants them:
//   MODE 0: plain, invalid rows -> 0      MODE 1: affine + activation on load, invalid rows -> 0
// `inf` is the group descriptor RowMapTC::info(r8) (the caller caches it per tile).
template <int MODE>
struct FeatSource {
    static constexpr bool USES_TMA = false;
    static constexpr bool SCATTER = false;
    RowMapTC rm;
    const __nv_bfloat16 *t;  // [C][ld]; MODE 1: the normalised value zhat, activation input is gamma*zhat+beta
    int C;
    int64_t ld;
    int act;
    int ones_line;  // channel index that carries 1 for valid rows (dW bias column), -1: none
    const float *gamma;
    const float *beta;
    int out_fmt;    // FMT_F16: forward operand; FMT_BF16: X side of a dW GEMM (meets bf16 gradients)
    __device__ __forceinline__ uint4 pack_out(const float (&f)[8]) const { return out_fmt == FMT_F16 ? pack8h(f) : pack8(f); }
    __device__ __forceinline__ void resolve(int64_t r) { rm.resolve(r); }
    __device__ __forceinline__ uint4 chunk_i(int ch, int64_t r8, unsigned inf) const
    {
        const int nv = gi_nv(inf);
        float f[8];
        if (ch == ones_line) {
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = e < nv ? 1.f : 0.f;
            return pack_out(f);
        }
        const bool live = ch < C && nv > 0;
        uint4 raw = make_uint4(0u, 0u, 0u, 0u);
        if (!live) return raw;
        raw = __ldg(reinterpret_cast<const uint4 *>(t + (int64_t)ch * ld + r8));
        if (MODE == 0 && nv == 8 && out_fmt == FMT_F16) return raw;
        unpack8h(raw, f);
        float ga = 1.f, be = 0.f;
        if (MODE != 0) {
            ga = gamma[ch];
            be = beta[ch];
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float v = f[e];
            if (MODE != 0) {
                v = fmaf(v, ga, be);
                if (act == B2PN_ACT_RELU) v = fmaxf(v, 0.f);
            }
            f[e] = e < nv ? v : 0.f;
        }
        return pack_out(f);
    }
};

// Y side of the dW GEMM fetched by TMA (a stored feature-major tensor whose invalid rows are already zero, e.g. dh after
// the BatchNorm-backward pass): the kernel issues the tensor-map copies itself, this only carries the row structure.
struct TmaSource {
    static constexpr bool USES_TMA = true;
    static constexpr bool SCATTER = false;
    RowMapTC rm;
    __device__ __forceinline__ void resolve(int64_t r) { rm.resolve(r); }
};

// The routed gradient of the max aggregation (SLOTS levels), generated on the fly instead of being stored:
//   dh3[ch][row] = dout[m][ch] if row is the arg-max slot of (centroid m, ch), else 0
// -- one value per (centroid, channel), i.e. 1 element in ~20..60 of the dense [c3][rows] tensor.  A chunk (8 rows of
// one channel) costs two L2-resident loads (arg, dout) in a loader thread; the dense tensor cost c3 * rows * 2 bytes of
// HBM written once and read twice per level.
struct RouteSource {
    static constexpr bool USES_TMA = false;
    RowMapTC rm;
    const float *dout;   // [n_dst][C]
    const int32_t *arg;  // [n_dst][C] arg-max slot
    int C;
    __device__ __forceinline__ void resolve(int64_t r) { rm.resolve(r); }
    static constexpr bool SCATTER = true;
    // The tile is zeros except for one element per (centroid that starts in it, channel): a centroid never crosses a
    // 64-row boundary, so its arg-max row is g*8 + arg inside the 64-row block its first row group g lies in.
    // A loader group zeroes the tile with 16-byte stores, meets at a named barrier, then every thread drops QUADS -- 4
    // consecutive channels of one centroid, one 16-byte load of arg and one of dout -- at their arg-max rows.  An item costs a thread ~100 instructions instead of the ~650 of a per-line fill
    // (ncu, round 2: with one loader warp per scheduler the routed kernels were bound by the loaders' dependent issue
    // latency, ~1.5 us per item, while the epilogue warps sat at their barrier 80 % of the time).
    // Needs C % 4 == 0 and 16-byte aligned arg / dout rows (`vec`, checked on the host); else four scalar loads.
    int vec;
    struct Quad {
        int4 a;
        float4 d;
    };
    __device__ __forceinline__ bool starts(unsigned inf, int ch4) const { return ch4 < C && gi_nv(inf) > 0 && gi_slot0(inf) == 0; }
    __device__ __forceinline__ void load_quad(unsigned inf, int ch4, Quad &q) const
    {
        const bool first = starts(inf, ch4);
        const int64_t idx = first ? (int64_t)gi_seg(inf) * C + ch4 : 0;
        if (vec) {
            q.a = __ldg(reinterpret_cast<const int4 *>(arg + idx));
            q.d = __ldg(reinterpret_cast<const float4 *>(dout + idx));
        } else {
            const int64_t last = (first ? (int64_t)gi_seg(inf) * C : 0) + C - 1;  // clamp inside the centroid's row
            q.a = make_int4(__ldg(arg + idx), __ldg(arg + min(idx + 1, last)), __ldg(arg + min(idx + 2, last)), __ldg(arg + min(idx + 3, last)));
            q.d = make_float4(__ldg(dout + idx), __ldg(dout + min(idx + 1, last)), __ldg(dout + min(idx + 2, last)),
                              __ldg(dout + min(idx + 3, last)));
        }
    }
    // lines l0 .. l0+3 (channels ch4 .. ch4+3) of the 64-row block at shared address `blk` (1024-byte aligned), row group g
    __device__ __forceinline__ void store_quad(const Quad &q, bool first, int ch4, int g, uint32_t blk, int l0) const
    {
        const int a[4] = {q.a.x, q.a.y, q.a.z, q.a.w};
        const float d[4] = {q.d.x, q.d.y, q.d.z, q.d.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const unsigned row = (unsigned)(g * 8 + a[e]);
            const unsigned ok = (first && ch4 + e < C && a[e] >= 0 && row < 64u) ? 1u : 0u;
            const uint32_t line = (uint32_t)(l0 + e);
            const uint32_t addr = blk + line * LINE_BYTES + ((((row >> 3) & 7u) ^ (line & 7u)) << 4) + ((row & 7u) << 1);
            const unsigned short gb = __bfloat16_as_ushort(__float2bfloat16(d[e]));
            asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p st.shared.b16 [%0], %1;\n\t}" ::"r"(addr), "h"(gb), "r"(ok)
                         : "memory");
        }
    }
    // my share of zeroing `bytes` (a multiple of 2048) at `base`: conflict-free 16-byte stores
    template <int NTHR = NUM_LOAD>
    static __device__ __forceinline__ void zero_tile(uint32_t base, int bytes, int lt)
    {
        for (int o = lt * 16; o < bytes; o += NTHR * 16)
            asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(base + (uint32_t)o), "r"(0u) : "memory");
    }
    template <int NTHR = NUM_LOAD>
    static __device__ __forceinline__ void group_barrier(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(NTHR) : "memory"); }
};

// MN-major B tile of the rows GEMM from a feature-major source: [2 row blocks of 64][64 channel lines];
// thread lt fills channel line (lt >> 1) of the chunk for row block (lt & 1)
// WIDE_: run under the wide kernel layout (two epilogue groups + one loader group, see tc_rows_gemm_kernel)
template <class SRC, bool WIDE_ = false>
struct FeatLoaderTC {
    static constexpr bool B_MN = true;
    static constexpr bool USES_TMA = false;
    static constexpr bool WIDE = WIDE_;
    // SCATTER sources (the routed gradient): the kernel runs the loader group as a software pipeline over quads (see
    // RouteSource) -- thread lt owns channel quad (lt & 15) of the 64-channel chunk and row group (lt >> 4) of both 64-row
    // blocks; descriptors are fetched one tile ahead, the (arg, dout) quads one item ahead of the shared-memory stores
    static constexpr bool PIPELINED = SRC::SCATTER;
    SRC src;
    int64_t row0;
    unsigned inf[8];  // descriptors of the 8 row groups of my row block
    // PIPELINED: TWO loader groups of 128 threads (8 warps) that take alternate items -- an item is a dependent chain
    // (descriptor -> quad loads -> zero fill -> group barrier -> scatter stores -> arrive), so one group alone leaves the
    // MMA and epilogue warps waiting however few instructions the chain has; two chains in flight halve the item period.
    // Thread lt of a group owns channel quad lt & 15 and row group lt >> 4 of both 64-row blocks.
    // Descriptors of my row group -- this tile (normalised), the next and the one after (RAW table words + a "past the
    // end" mask: normalising would wait for the load right where it is issued)
    static constexpr int PIPE_GROUPS = 2;
    unsigned qinf[2], qraw1[2], qraw2[2], qdead1, qdead2;
    struct Item {
        typename SRC::Quad q[2];
        unsigned first;  // bit b: a centroid starts in my row group of row block b (known without waiting for the loads)
    };
    __device__ __forceinline__ void resolve(int64_t r) { src.resolve(r); }
    // request the descriptors of `tile` (SLOTS levels only: routed gradients exist nowhere else)
    __device__ __forceinline__ void fetch_tile(int64_t tile, int lt)
    {
        const int64_t r0 = tile * R + (lt >> 4) * 8;
        qdead2 = 0u;
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            const int64_t r8 = r0 + b * 64;
            qraw2[b] = __ldg(src.rm.rgrp + (r8 >> 3));
            qdead2 |= (r8 >= src.rm.rows ? 1u : 0u) << b;
        }
    }
    __device__ __forceinline__ void no_tile() { qraw2[0] = qraw2[1] = GI_NONE, qdead2 = 3u; }
    // the tile after next becomes the next one
    __device__ __forceinline__ void shift_tiles()
    {
#pragma unroll
        for (int b = 0; b < 2; ++b) qraw1[b] = qraw2[b];
        qdead1 = qdead2;
    }
    // the next tile becomes the current one
    __device__ __forceinline__ void advance_tile()
    {
#pragma unroll
        for (int b = 0; b < 2; ++b) qinf[b] = (((qdead1 >> b) & 1u) || gi_none(qraw1[b])) ? GI_NONE : qraw1[b];
    }
    // pull the (arg, dout) rows the NEXT tile will read into L2 (each is read exactly once: a compulsory DRAM miss that a
    // one-item-ahead register prefetch cannot cover); two threads per 256 bytes of a chunk issue the prefetches
    __device__ __forceinline__ void prefetch_next_rows(int lt, int kc0, int kstep, int num_kc) const
    {
        if ((lt & 7) != 0) return;
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            const unsigned w = qraw1[b];
            if (((qdead1 >> b) & 1u) || gi_none(w) || gi_nv(w) == 0 || gi_slot0(w) != 0) continue;
            const int64_t base = (int64_t)gi_seg(w) * src.C + (lt & 15) * 4;
            for (int kc = kc0; kc < num_kc; kc += kstep) {
                if (kc * KC + (lt & 15) * 4 >= src.C) break;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(src.arg + base + kc * KC));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(src.dout + base + kc * KC));
            }
        }
    }
    __device__ __forceinline__ void load(int kc, int lt, Item &it) const
    {
        const int ch4 = kc * KC + (lt & 15) * 4;
        it.first = 0u;
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            src.load_quad(qinf[b], ch4, it.q[b]);
            it.first |= (src.starts(qinf[b], ch4) ? 1u : 0u) << b;
        }
    }
    // after the group has zeroed the tile and met at its barrier
    __device__ __forceinline__ void store(uint8_t *B, int kc, int lt, const Item &it) const
    {
        const int ch4 = kc * KC + (lt & 15) * 4;
#pragma unroll
        for (int b = 0; b < 2; ++b)
            src.store_quad(it.q[b], (it.first >> b) & 1u, ch4, lt >> 4, smem_u32(B) + b * (64 * LINE_BYTES), (lt & 15) * 4);
    }
    __device__ __forceinline__ void begin_tile(int64_t tile, int lt)
    {
        row0 = tile * R + (lt & 1) * 64;
        if (src.rm.seg_mode) {
#pragma unroll
            for (int g = 0; g < 8; ++g) inf[g] = src.rm.info(row0 + g * 8);
        } else {
#pragma unroll
            for (int g = 0; g < 8; ++g) inf[g] = src.rm.info_slots(row0 + g * 8);
        }
    }
    __device__ __forceinline__ void produce(uint8_t *B, int kc, int lt) const
    {
        const int cl = lt >> 1, nb = lt & 1;
        uint8_t *dst = B + nb * (64 * LINE_BYTES);
        const int ch = kc * KC + cl;
        uint4 v[8];
#pragma unroll
        for (int g = 0; g < 8; ++g) v[g] = src.chunk_i(ch, row0 + g * 8, inf[g]);
#pragma unroll
        for (int g = 0; g < 8; ++g) *reinterpret_cast<uint4 *>(dst + line_chunk_off(cl, g)) = v[g];
    }
    // MN-major: 16 k lines per step; LBO = stride between the two 64-row blocks, SBO = 8 lines
    static __device__ __forceinline__ uint64_t b_desc(uint32_t b_saddr, int ks)
    {
        return smem_desc_sw128(b_saddr + ks * (16 * LINE_BYTES), 64 * LINE_BYTES, ATOM_BYTES);
    }
};

// The same MN-major B tile fetched by the TMA unit: for a stored feature-major tensor that needs no arithmetic on
// the way in (invalid rows already zero) the whole tile is two tensor-map copies issued by one thread -- no loader
// instructions, no registers, any prefetch depth the stage ring allows.
struct TmaFeatLoader {
    static constexpr bool B_MN = true;
    static constexpr bool USES_TMA = true;
    static constexpr bool WIDE = true;
    __device__ __forceinline__ void resolve(int64_t) {}
    __device__ __forceinline__ void begin_tile(int64_t, int) {}
    __device__ __forceinline__ void produce_tma(uint8_t *B, int64_t tile, int kc, const TmaMap *map, uint64_t *bar) const
    {
        mbar_expect_tx(bar, B_BYTES);
        tma_load_2d(B, map, (int)(tile * R), kc * KC, bar);
        tma_load_2d(B + 64 * LINE_BYTES, map, (int)(tile * R + 64), kc * KC, bar);
    }
    static __device__ __forceinline__ uint64_t b_desc(uint32_t b_saddr, int ks)
    {
        return smem_desc_sw128(b_saddr + ks * (16 * LINE_BYTES), 64 * LINE_BYTES, ATOM_BYTES);
    }
};

// =================================================================================================
//  Epilogues of the rows GEMM (128 threads; thread tid owns TMEM lane tid = channel within the M tile)
// =================================================================================================
// what the kernel hands an epilogue per call: the warp's shared-memory staging area (two 32-line x 128-byte tiles,
// only for STAGED epilogues) and the tensor maps their TMA stores go through
struct EpCtx {
    uint8_t *stage;
    const TmaMap *m0;
    const TmaMap *m1;
    uint64_t *bar;       // the warp's own mbarrier (TMA loads into the staging area)
    int64_t next_tile;   // the (tile, mt) this thread's epilogue handles after the current one, -1: none
    int next_ch;         // its channel for this thread
};
constexpr int EPI_STAGE_PER_WARP = 2 * 32 * LINE_BYTES;  // 8 KB

// a STAGED epilogue thread owns one channel = one 128-byte line of 64 rows: it writes the line (swizzled like every
// other tile here) into the warp's staging tile and one lane sends the 32 x 64 tile out with a single TMA store --
// 16-byte global stores 2*ld bytes apart per lane (32 lines per instruction) were what these epilogues spent their time on
__device__ __forceinline__ void stage_chunk(uint8_t *tile32, int lane, int g, const uint4 &v)
{
    *reinterpret_cast<uint4 *>(tile32 + lane * LINE_BYTES + ((g ^ (lane & 7)) << 4)) = v;
}
__device__ __forceinline__ uint4 unstage_chunk(const uint8_t *tile32, int lane, int g)
{
    return *reinterpret_cast<const uint4 *>(tile32 + lane * LINE_BYTES + ((g ^ (lane & 7)) << 4));
}

struct StoreF32Ep {  // self-test: out[ch][row] = acc
    static constexpr bool STAGED = false;
    float *out;
    int C;
    int64_t ld;
    __device__ __forceinline__ void resolve(int64_t) {}
    __device__ __forceinline__ void begin() {}
    __device__ __forceinline__ void tile_mt(uint32_t taddr, int64_t tile, int ch, int mt, int half, const EpCtx &cx)
    {
#pragma unroll 1
        for (int cc = half * 2; cc < half * 2 + 2; ++cc) {
            float v[32];
            tmem_ld32(taddr + cc * 32, v);
            if (ch < C) {
                float4 *dst = reinterpret_cast<float4 *>(out + (int64_t)ch * ld + tile * R + cc * 32);
#pragma unroll
                for (int j = 0; j < 8; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
        }
    }
    __device__ __forceinline__ void finish_mt(int ch, int mt, int half) {}
};

template <int MT>
struct StatsEpTC {  // pass A of a BatchNorm layer: per-channel sum and sum of squares of the bias-free accumulators
    static constexpr bool STAGED = false;
    int C;
    double *partial;  // [gridDim.x * nslot][2][cpad]
    int cpad;
    int nslot;        // epilogue thread groups per CTA writing partials (2 column halves x epilogue groups)
    double S[MT], Q[MT];
    __device__ __forceinline__ void resolve(int64_t) {}
    __device__ __forceinline__ void begin()
    {
#pragma unroll
        for (int i = 0; i < MT; ++i) S[i] = Q[i] = 0.0;
    }
    __device__ __forceinline__ void tile_mt(uint32_t taddr, int64_t tile, int ch, int mt, int half, const EpCtx &cx)
    {
        float s = 0.f, q = 0.f;
#pragma unroll 1
        for (int cc = half * 2; cc < half * 2 + 2; ++cc) {
            float v[32];
            tmem_ld32(taddr + cc * 32, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                s += v[j];
                q = fmaf(v[j], v[j], q);
            }
        }
        S[mt] += (double)s;
        Q[mt] += (double)q;
    }
    __device__ __forceinline__ void finish_mt(int ch, int mt, int slot)
    {
        if (ch < C) {
            double *pt = partial + ((int64_t)blockIdx.x * nslot + slot) * 2 * cpad;
            pt[ch] = S[mt];
            pt[cpad + ch] = Q[mt];
        }
    }
};

struct NormStoreEpTC {  // pass B: zT[ch][row] = fp16((acc + bias - mean) * rstd), the NORMALISED value zhat (what backward
                        // needs), and aT[ch][row] = fp16(act(gamma*zhat + beta)) with invalid rows zeroed: the operand
                        // of the next layer and of the dW GEMMs, stored so that they can take it through the TMA unit
    static constexpr bool STAGED = true;
    // zT and aT leave through the warp's staging tiles and two TMA stores (EpCtx::m0 = map of z, m1 = map of a)
    int C;
    const float *bias;
    const float *mean;
    const float *rstd;
    const float *gamma;
    const float *beta;
    int act;
    RowMapTC rm;
    __device__ __forceinline__ void resolve(int64_t r) { rm.resolve(r); }
    __device__ __forceinline__ void begin() {}
    __device__ __forceinline__ void tile_mt(uint32_t taddr, int64_t tile, int ch, int mt, int half, const EpCtx &cx)
    {
        const int lane = threadIdx.x & 31;
        float sc = 0.f, sh = 0.f, ga = 0.f, be = 0.f;
        if (ch < C) {
            sc = rstd[ch];
            sh = (bias[ch] - mean[ch]) * sc;
            ga = gamma[ch];
            be = beta[ch];
        }
        uint8_t *zt = cx.stage, *at = cx.stage + 32 * LINE_BYTES;
        const unsigned nv64 = rm.valid64(tile * R + half * 64);  // valid rows of my eight 8-row groups (warp-uniform)
        if (lane == 0) bulk_wait_read_all();  // the TMA stores of my previous tile have read the staging tiles
        __syncwarp();
#pragma unroll 1
        for (int cc = half * 2; cc < half * 2 + 2; ++cc) {
            float v[32];
            tmem_ld32(taddr + cc * 32, v);
            const unsigned nvs = nv64 >> (16 * (cc - half * 2));
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int nv = (int)((nvs >> (4 * j)) & 15u);
                float f[8], g[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) f[e] = fmaf(v[8 * j + e], sc, sh);
                const uint4 zp = pack8h(f);
                unpack8h(zp, f);  // the activation is defined on the STORED (fp16) zhat, as backward recomputes it
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    float y = fmaf(f[e], ga, be);
                    if (act == B2PN_ACT_RELU) y = fmaxf(y, 0.f);
                    g[e] = e < nv ? y : 0.f;
                }
                const int gidx = (cc - half * 2) * 4 + j;  // 16-byte chunk of my 128-byte line (64 rows of this half)
                stage_chunk(zt, lane, gidx, zp);
                stage_chunk(at, lane, gidx, pack8h(g));
            }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {  // channels past C are clipped by the tensor map
            const int x = (int)(tile * R + half * 64), y = ch;  // lane 0's channel = first of the warp's 32
            tma_store_2d(cx.m0, zt, x, y);
            tma_store_2d(cx.m1, at, x, y);
            bulk_commit_group();
        }
    }
    __device__ __forceinline__ void finish_mt(int ch, int mt, int half)
    {
        if ((threadIdx.x & 31) == 0) bulk_wait_all();
    }
};

struct SlotMaxEpTC {  // out[m][ch] = max over the valid rows of centroid m, arg = first max SLOT (compacted rows:
                      // a centroid is a run of 8-row groups that never crosses a 64-row boundary)
    static constexpr bool STAGED = false;
    float *out;  // [n_dst][C] fp32 row-major
    int32_t *arg;
    int C;
    const float *bias;
    const uint32_t *rgrp;
    int64_t rows;
    __half *out16;  // optional fp16 copy of out (the next level's gather operand)
    __device__ __forceinline__ void resolve(int64_t r) { rows = r; }
    __device__ __forceinline__ void begin() {}
    __device__ __forceinline__ void tile_mt(uint32_t taddr, int64_t tile, int ch, int mt, int half, const EpCtx &cx)
    {
        const float b = ch < C ? bias[ch] : 0.f;
        float best = -INFINITY;
        int bk = -1;
#pragma unroll 1
        for (int cc = half * 2; cc < half * 2 + 2; ++cc) {
            float v[32];
            tmem_ld32(taddr + cc * 32, v);
            const int64_t g0 = tile * (R / 8) + cc * 4;
#pragma unroll
            for (int gg = 0; gg < 4; ++gg) {
                unsigned inf = GI_NONE;
                if ((g0 + gg) * 8 < rows) inf = __ldg(rgrp + g0 + gg);  // warp-uniform
                if (gi_none(inf)) continue;
                const int s0 = gi_slot0(inf), nv = gi_nv(inf);
                if (s0 == 0) {
                    best = -INFINITY;
                    bk = -1;
                }
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const float x = v[gg * 8 + e] + b;
                    if (e < nv && x > best) {
                        best = x;
                        bk = s0 + e;
                    }
                }
                if (gi_last(inf) && ch < C) {
                    const int64_t m = gi_seg(inf);
                    const float o = bk >= 0 ? best : 0.f;
                    out[m * C + ch] = o;
                    arg[m * C + ch] = bk;
                    if (out16) out16[m * C + ch] = __float2half_rn(o);
                }
            }
        }
    }
    __device__ __forceinline__ void finish_mt(int ch, int mt, int half) {}
};

__device__ __forceinline__ unsigned f32_orderable_tc(float f)
{
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

struct CloudMaxEpTC {  // global_max_pool over sorted cloud ids: 64-bit atomicMax keys, unpacked by a tiny kernel
    static constexpr bool STAGED = false;
    unsigned long long *keys;  // [n_dst][C], zero-initialised
    int C;
    const float *bias;
    const int64_t *batch;
    int64_t rows;
    __device__ __forceinline__ void resolve(int64_t) {}
    __device__ __forceinline__ void begin() {}
    __device__ __forceinline__ void tile_mt(uint32_t taddr, int64_t tile, int ch, int mt, int half, const EpCtx &cx)
    {
        const float b = ch < C ? bias[ch] : 0.f;
        int64_t curseg = -1;
        unsigned long long best = 0ull;
#pragma unroll 1
        for (int cc = half * 2; cc < half * 2 + 2; ++cc) {
            float v[32];
            tmem_ld32(taddr + cc * 32, v);
            if (ch < C) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int64_t row = tile * R + cc * 32 + j;
                    if (row < rows) {
                        const int64_t sg = batch[row];
                        if (sg != curseg) {
                            if (curseg >= 0) atomicMax(keys + curseg * C + ch, best);
                            curseg = sg;
                            best = 0ull;
                        }
                        const unsigned long long key = ((unsigned long long)f32_orderable_tc(v[j] + b) << 32) |
                                                       (unsigned long long)(0xffffffffu - (unsigned)row);
                        best = key > best ? key : best;
                    }
                }
            }
        }
        if (ch < C && curseg >= 0) atomicMax(keys + curseg * C + ch, best);
    }
    __device__ __forceinline__ void finish_mt(int ch, int mt, int half) {}
};

template <int MT>
struct MaskSumsStoreEpTC {  // backward through activation + sums for the BatchNorm backward (thread = channel of the
                            // layer being differentiated through): dz = da * [z > 0];  S1 = sum dz, S2 = sum dz * zhat
    static constexpr bool STAGED = true;
    // zhat arrives and dz leaves through the warp's staging tiles: one TMA load (prefetched a tile ahead) and one TMA
    // store per warp and tile instead of 16 global accesses per thread, 2*ld bytes apart per lane
    int C;
    const float *gamma;
    const float *beta;
    int act;
    double *partial;
    int cpad;
    int nslot;
    double S[MT], Q[MT];
    unsigned phase;
    bool primed;
    __device__ __forceinline__ void resolve(int64_t) {}
    __device__ __forceinline__ void begin()
    {
#pragma unroll
        for (int i = 0; i < MT; ++i) S[i] = Q[i] = 0.0;
        phase = 0u;
        primed = false;
    }
    static __device__ __forceinline__ void fetch_z(const EpCtx &cx, uint8_t *zt, int64_t tile, int ch0, int half)
    {
        mbar_arrive_expect_tx(cx.bar, 32 * LINE_BYTES);
        tma_load_2d(zt, cx.m1, (int)(tile * R + half * 64), ch0, cx.bar);
    }
    __device__ __forceinline__ void tile_mt(uint32_t taddr, int64_t tile, int ch, int mt, int half, const EpCtx &cx)
    {
        const int lane = threadIdx.x & 31;
        uint8_t *dt = cx.stage, *zt = cx.stage + 32 * LINE_BYTES;
        if (!primed) {  // first tile of this warp: nothing was prefetched yet
            if (lane == 0) fetch_z(cx, zt, tile, ch, half);
            primed = true;
        }
        float be = 0.f, ga = 0.f;
        if (ch < C) {
            be = beta[ch];
            ga = gamma[ch];
        }
        if (lane == 0) bulk_wait_read_all();  // my previous dz store has read its staging tile
        __syncwarp();
        mbar_wait(cx.bar, phase);  // zhat tile landed
        phase ^= 1u;
        float s = 0.f, q = 0.f;
        const bool relu = act == B2PN_ACT_RELU;
#pragma unroll 1
        for (int cc = half * 2; cc < half * 2 + 2; ++cc) {
            float v[32];
            tmem_ld32(taddr + cc * 32, v);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int gidx = (cc - half * 2) * 4 + j;
                float zf[8], o[8];
                unpack8h(unstage_chunk(zt, lane, gidx), zf);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    // channels past C: zero-padded weight rows give da = 0 exactly (and ga = be = 0 mask them under ReLU);
                    // invalid rows: da = 0 because their operand columns are zero
                    const float da = v[8 * j + e];
                    const float g = (!relu || fmaf(zf[e], ga, be) > 0.f) ? da : 0.f;
                    s += g;
                    q = fmaf(g, zf[e], q);
                    o[e] = g;
                }
                stage_chunk(dt, lane, gidx, pack8(o));
            }
        }
        S[mt] += (double)s;
        Q[mt] += (double)q;
        fence_proxy_async_smem();
        __syncwarp();  // everybody has read zt and written dt
        if (lane == 0) {
            tma_store_2d(cx.m0, dt, (int)(tile * R + half * 64), ch);
            bulk_commit_group();
            if (cx.next_tile >= 0) fetch_z(cx, zt, cx.next_tile, cx.next_ch, half);
        }
    }
    __device__ __forceinline__ void finish_mt(int ch, int mt, int slot)
    {
        if ((threadIdx.x & 31) == 0) bulk_wait_all();
        if (ch < C) {
            double *pt = partial + ((int64_t)blockIdx.x * nslot + slot) * 2 * cpad;
            pt[ch] = S[mt];
            pt[cpad + ch] = Q[mt];
        }
    }
};

constexpr float FIXED_ONE = 1099511627776.f;  // 2^40: fixed-point unit of the deterministic scatter accumulator
__global__ void fixed_to_f32_kernel(const long long *acc, float *out, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)((double)acc[i] * (1.0 / 1099511627776.0));
}

struct ScatterEpTC {  // gradient w.r.t. the gathered source features
    // A thread drains one channel (TMEM lane) over 64 rows, but dx is row-major [n_src][C]: the warp transposes its
    // 32 channels x 64 rows through its staging tile (fp32, swizzled per float4), after which a lane owns a ROW and
    // adds four consecutive channels per instruction (red.global.add.v4.f32: a quarter of the atomic operations the
    // channel-per-thread form needed; CLOUDS levels: plain 16-byte stores).
    // Deterministic mode (b2pn_sa_args::deterministic, SLOTS levels): the addends go into a 64-bit FIXED-POINT
    // accumulator (2^-40 units) with integer atomics -- integer addition is associative, so the sums do not depend on the
    // order in which the rows arrive -- and fixed_to_f32_kernel converts the result; bit-reproducible feature gradients.
    static constexpr bool STAGED = true;
    RowMapTC rm;
    float *dx;  // [n_src][C] fp32, zero-initialised by the caller in SLOTS mode
    int C;
    long long *dxi;  // [n_src][C] fixed-point accumulator (zeroed), or NULL: fp32 atomics straight into dx
    __device__ __forceinline__ void resolve(int64_t rows) { rm.rows = rows; }
    __device__ __forceinline__ void begin() {}
    __device__ __forceinline__ void tile_mt(uint32_t taddr, int64_t tile, int ch, int mt, int half, const EpCtx &cx)
    {
        const int lane = threadIdx.x & 31;
        const int ch0 = ch - lane;  // first channel of this warp
        float *st = reinterpret_cast<float *>(cx.stage);  // [64 rows][32 channels]
        __syncwarp();  // the previous tile's reads are done
#pragma unroll 1
        for (int cc = 0; cc < 2; ++cc) {
            float v[32];
            tmem_ld32(taddr + (half * 2 + cc) * 32, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int r = cc * 32 + j;
                st[r * 32 + ((((lane >> 2) ^ (r & 7))) << 2) + (lane & 3)] = v[j];
            }
        }
        __syncwarp();
        const bool vec = (C & 3) == 0;
#pragma unroll 1
        for (int rr = 0; rr < 2; ++rr) {
            const int r = rr * 32 + lane;
            const int64_t row = tile * R + half * 64 + r;
            if (row >= rm.rows) continue;
            int64_t dst = row;
            if (!rm.seg_mode) {
                const int sidx = __ldg(rm.row_src + row);
                if (sidx < 0) continue;
                dst = sidx;
            }
            float *base = dx + dst * C + ch0;
#pragma unroll
            for (int c4 = 0; c4 < 8; ++c4) {
                if (ch0 + c4 * 4 >= C) break;
                const float4 q = *reinterpret_cast<const float4 *>(st + r * 32 + ((c4 ^ (r & 7)) << 2));
                if (dxi != nullptr && !rm.seg_mode) {
                    const float e[4] = {q.x, q.y, q.z, q.w};
                    unsigned long long *acc = reinterpret_cast<unsigned long long *>(dxi + dst * C + ch0 + c4 * 4);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (ch0 + c4 * 4 + k >= C) break;
                        if (e[k] != 0.f) atomicAdd(acc + k, (unsigned long long)__float2ll_rn(e[k] * FIXED_ONE));
                    }
                } else if (vec) {
                    if (rm.seg_mode) {
                        *reinterpret_cast<float4 *>(base + c4 * 4) = q;
                    } else if (q.x != 0.f || q.y != 0.f || q.z != 0.f || q.w != 0.f) {
                        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(base + c4 * 4), "f"(q.x), "f"(q.y), "f"(q.z),
                                     "f"(q.w)
                                     : "memory");
                    }
                } else {
                    const float e[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (ch0 + c4 * 4 + k >= C) break;
                        if (rm.seg_mode) base[c4 * 4 + k] = e[k];
                        else if (e[k] != 0.f) atomicAdd(base + c4 * 4 + k, e[k]);
                    }
                }
            }
        }
    }
    __device__ __forceinline__ void finish_mt(int ch, int mt, int half) {}
};

// =================================================================================================
//  The rows GEMM kernel:  D^T[channel, row] = A[channel, k] * B[k, row]
// =================================================================================================
template <int MT, bool STAGED, bool TMA>
struct SmemPlan {
    static constexpr int A_BYTES = MT * 128 * LINE_BYTES;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int EPI_WARPS = (TMA ? 2 : 1) * (NUM_EPI / 32);
    // the epilogue staging tiles (8 KB per epilogue warp) come out of the operand ring
    static constexpr int STAGES = !STAGED ? (MT == 1 ? 5 : 4) : (TMA ? (MT == 1 ? 3 : 2) : (MT == 1 ? 4 : 3));
    static constexpr int EPI_OFF = STAGES * STAGE_BYTES;
    static constexpr int EPI_BYTES = STAGED ? EPI_WARPS * EPI_STAGE_PER_WARP : 0;
    static constexpr int BAR_OFF = EPI_OFF + EPI_BYTES;
    static constexpr int TOTAL = BAR_OFF + 256 + 1024;  // barriers + alignment slack
};

template <class BL, class = void>
struct LoaderPipelined { static constexpr bool value = false; };
template <class BL>
struct LoaderPipelined<BL, decltype((void)BL::PIPELINED)> { static constexpr bool value = BL::PIPELINED; };

template <class BL, class = void>
struct LoaderGroupsWide { static constexpr int value = 1; };   // loader groups under the wide layout
template <class BL>
struct LoaderGroupsWide<BL, decltype((void)BL::PIPE_GROUPS)> { static constexpr int value = BL::PIPELINED ? BL::PIPE_GROUPS : 1; };
template <class BL>
constexpr int gemm_threads() { return BL::USES_TMA ? NT_TMA : (BL::WIDE ? NT_WIDE + (LoaderGroupsWide<BL>::value - 1) * NUM_LOAD : NT); }

template <int MT, class BL, class EP>
__global__ void __launch_bounds__(gemm_threads<BL>(), 1)
    tc_rows_gemm_kernel(const GemmParams gp, BL bl, EP ep, const __grid_constant__ TmaMap tmap, const __grid_constant__ TmaMap tmap_e0,
                        const __grid_constant__ TmaMap tmap_e1)
{
    constexpr bool TMA = BL::USES_TMA;
    constexpr bool WIDE = BL::WIDE;
    static_assert(!TMA || WIDE, "TMA-fed kernels use the wide layout");
    constexpr int EPI_GROUPS = WIDE ? 2 : 1;
    constexpr int EPI_WARPS = EPI_GROUPS * (NUM_EPI / 32);
    // SIMT loaders: two groups in warps 8-15 (narrow layout) or one group in warps 17-20 (wide layout)
    constexpr int LGROUPS = WIDE ? LoaderGroupsWide<BL>::value : LOAD_GROUPS;
    constexpr int LOAD_T0 = WIDE ? (MMA_WARP + 1) * 32 : NUM_EPI;
    constexpr int NLOAD = NUM_LOAD;  // threads of a SIMT loader group
    using P = SmemPlan<MT, EP::STAGED, WIDE>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + P::BAR_OFF);
    uint64_t *empty = full + P::STAGES;
    uint64_t *tfull = empty + P::STAGES;
    uint64_t *tempty = tfull + 2;
    uint64_t *ebar = tempty + 2;  // one per epilogue warp
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(ebar + EPI_WARPS);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int mg = blockIdx.y;
    constexpr int TCOLS = MT * R * 2;  // two accumulator buffers
    const int64_t rows = gp.rows_dev ? *gp.rows_dev : gp.rows;
    const int64_t num_tiles = (rows + R - 1) / R;
    bl.resolve(rows);
    ep.resolve(rows);

    if (tid == 0) {
        for (int s = 0; s < P::STAGES; ++s) {
            mbar_init(&full[s], TMA ? 1 : NLOAD);
            mbar_init(&empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull[a], 1);
            mbar_init(&tempty[a], NUM_EPI);
        }
        for (int w = 0; w < EPI_WARPS; ++w) mbar_init(&ebar[w], 1);
        fence_barrier_init();
    }
    if (warp == MMA_WARP) tmem_alloc<TCOLS>(tmem_holder);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    if (TMA && warp == PROD_WARP_TMA) {
        // ------------------------------------------------------------------ producer: one thread, TMA only
        if constexpr (TMA) {
            if (lane == 0) {
                uint32_t it = 0;
                for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                    for (int kc = 0; kc < gp.num_kc; ++kc, ++it) {
                        const int s = it % P::STAGES;
                        const uint32_t ph = (it / P::STAGES) & 1u;
                        mbar_wait(&empty[s], ph ^ 1u);
                        uint8_t *A = smem + s * P::STAGE_BYTES;
                        uint8_t *B = A + P::A_BYTES;
                        mbar_expect_tx(&full[s], P::A_BYTES);
                        bulk_g2s(A, gp.a_packed + ((int64_t)mg * gp.num_kc + kc) * P::A_BYTES, P::A_BYTES, &full[s]);
                        bl.produce_tma(B, tile, kc, &tmap, &full[s]);
                        mbar_arrive(&full[s]);
                    }
                }
            }
        }
    } else if (!TMA && tid >= LOAD_T0 && tid < LOAD_T0 + LGROUPS * NLOAD) {
        // ------------------------------------------------------------------ SIMT loaders: group g takes every
        // LGROUPS-th (tile, k-chunk) item, so the groups' global-load latencies overlap
        if constexpr (!TMA) {
            const int g = (tid - LOAD_T0) / NLOAD;
            const int lt = (tid - LOAD_T0) % NLOAD;
            if constexpr (LoaderPipelined<BL>::value) {
                // group g takes items g, g + LGROUPS, ... of this CTA's (tile, k-chunk) sequence
                typename BL::Item cur, nxt;
                const int num_kc = gp.num_kc;
                const int64_t my_tiles = blockIdx.x < num_tiles ? (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
                const int64_t items = my_tiles * num_kc;
                const int tstep = num_kc >= LGROUPS ? 1 : LGROUPS / num_kc;  // my tile sequence: every tile, or every tstep-th
                auto tile_of = [&](int64_t tl) { return (int64_t)blockIdx.x + tl * gridDim.x; };
                auto fetch_or_none = [&](int64_t tl) {
                    if (tl < my_tiles) bl.fetch_tile(tile_of(tl), lt);
                    else bl.no_tile();
                };
                int64_t i = g;
                if (i < items) {
                    int64_t tl = i / num_kc;
                    int kc = (int)(i % num_kc);
                    // descriptor pipeline: this tile / next / the one after
                    bl.fetch_tile(tile_of(tl), lt);
                    bl.shift_tiles();
                    bl.advance_tile();
                    bl.load(kc, lt, cur);
                    fetch_or_none(tl + tstep);
                    bl.shift_tiles();
                    bl.prefetch_next_rows(lt, num_kc % LGROUPS == 0 ? g : 0, num_kc % LGROUPS == 0 ? LGROUPS : 1, num_kc);
                    fetch_or_none(tl + 2 * tstep);
                    // one item: `c` holds its quads (requested one item ago), `n` receives the next item's.  Called with the
                    // two register sets swapped every other item -- a `cur = nxt` copy would wait for the loads in flight
                    auto item = [&](typename BL::Item &c, typename BL::Item &n) -> bool {
                        const int64_t ni = i + LGROUPS;
                        const bool has_next = ni < items;
                        int nkc = kc + LGROUPS;
                        int64_t ntl = tl;
                        while (nkc >= num_kc) {
                            nkc -= num_kc;
                            ++ntl;
                        }
                        if (has_next) {
                            if (ntl != tl) bl.advance_tile();
                            bl.load(nkc, lt, n);
                            if (ntl != tl) {
                                // entered a new tile: its successor's descriptors have landed -> pull its rows into L2, and
                                // request the descriptors of the tile after that
                                bl.shift_tiles();
                                bl.prefetch_next_rows(lt, num_kc % LGROUPS == 0 ? g : 0, num_kc % LGROUPS == 0 ? LGROUPS : 1, num_kc);
                                fetch_or_none(ntl + 2 * tstep);
                            }
                        }
                        const int s = (int)(i % P::STAGES);
                        const uint32_t ph = (uint32_t)(i / P::STAGES) & 1u;
                        mbar_wait(&empty[s], ph ^ 1u);
                        uint8_t *A = smem + s * P::STAGE_BYTES;
                        uint8_t *B = A + P::A_BYTES;
                        if (lt == 0) {
                            mbar_expect_tx(&full[s], P::A_BYTES);
                            bulk_g2s(A, gp.a_packed + ((int64_t)mg * num_kc + kc) * P::A_BYTES, P::A_BYTES, &full[s]);
                        }
                        RouteSource::zero_tile<NLOAD>(smem_u32(B), B_BYTES, lt);
                        RouteSource::group_barrier<NLOAD>(1 + g);
                        bl.store(B, kc, lt, c);
                        fence_proxy_async_smem();
                        mbar_arrive(&full[s]);
                        i = ni;
                        kc = nkc;
                        tl = ntl;
                        return has_next;
                    };
                    while (item(cur, nxt) && item(nxt, cur)) {
                    }
                }
            } else {
                uint32_t it = 0;
                int64_t cur_tile = -1;
                for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                    for (int kc = 0; kc < gp.num_kc; ++kc, ++it) {
                        if ((int)(it % LGROUPS) != g) continue;
                        if (tile != cur_tile) {
                            bl.begin_tile(tile, lt);
                            cur_tile = tile;
                        }
                        const int s = it % P::STAGES;
                        const uint32_t ph = (it / P::STAGES) & 1u;
                        mbar_wait(&empty[s], ph ^ 1u);
                        uint8_t *A = smem + s * P::STAGE_BYTES;
                        uint8_t *B = A + P::A_BYTES;
                        if (lt == 0) {
                            mbar_expect_tx(&full[s], P::A_BYTES);
                            bulk_g2s(A, gp.a_packed + ((int64_t)mg * gp.num_kc + kc) * P::A_BYTES, P::A_BYTES, &full[s]);
                        }
                        bl.produce(B, kc, lt);
                        fence_proxy_async_smem();
                        mbar_arrive(&full[s]);
                    }
                }
            }
        }
    } else if (warp == MMA_WARP) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t IDESC = idesc_16(128, R, false, BL::B_MN, gp.a_fmt, gp.b_fmt);
            uint32_t it = 0, tl = 0;
            for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++tl) {
                const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
                mbar_wait(&tempty[acc], aph ^ 1u);
                tc_fence_after();
                for (int kc = 0; kc < gp.num_kc; ++kc, ++it) {
                    const int s = it % P::STAGES;
                    const uint32_t ph = (it / P::STAGES) & 1u;
                    mbar_wait(&full[s], ph);
                    tc_fence_after();
                    const uint32_t a_s = smem_u32(smem + s * P::STAGE_BYTES);
                    const uint32_t b_s = a_s + P::A_BYTES;
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
                        for (int ks = 0; ks < KC / 16; ++ks) {
                            const uint64_t ad = smem_desc_sw128(a_s + mt * (128 * LINE_BYTES) + ks * 32, 16, ATOM_BYTES);
                            const uint64_t bd = BL::b_desc(b_s, ks);
                            umma_bf16(tmem_base + acc * (MT * R) + mt * R, ad, bd, IDESC, (kc | ks) != 0);
                        }
                    }
                    umma_commit(&empty[s]);
                }
                umma_commit(&tfull[acc]);
            }
        }
    } else if (warp < EPI_WARPS) {
        // ------------------------------------------------------------------ epilogue: group g = warp / 8 drains the
        // tiles with tl % EPI_GROUPS == g (with two groups: tile parity = accumulator buffer)
        ep.begin();
        const int grp = warp >> 3, w8 = warp & 7;
        const int half = w8 >> 2;
        const int chl = tid & 127;
        const uint32_t lane_base = ((uint32_t)((warp & 3) * 32)) << 16;
        EpCtx cx;
        cx.stage = smem + P::EPI_OFF + warp * EPI_STAGE_PER_WARP;
        cx.m0 = &tmap_e0;
        cx.m1 = &tmap_e1;
        cx.bar = &ebar[warp];
        const int64_t tstep = (int64_t)EPI_GROUPS * gridDim.x;
        uint32_t tl = (uint32_t)grp;
        for (int64_t tile = blockIdx.x + (int64_t)grp * gridDim.x; tile < num_tiles; tile += tstep, tl += EPI_GROUPS) {
            const uint32_t acc = tl & 1u, aph = (tl >> 1) & 1u;
            mbar_wait(&tfull[acc], aph);
            tc_fence_after();
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const int ch = (mg * MT + mt) * 128 + chl;
                if (mt + 1 < MT) {
                    cx.next_tile = tile;
                    cx.next_ch = ch + 128;
                } else {
                    cx.next_tile = tile + tstep < num_tiles ? tile + tstep : -1;
                    cx.next_ch = mg * MT * 128 + chl;
                }
                // a warp whose 32 channels all lie past the layer's width has nothing to drain (TMEM lane quarters are
                // tied to warp % 4, so it cannot help the others either): it only keeps the barrier protocol
                // (MT == 1 only: with two M tiles a staged epilogue prefetches across them)
                if (MT > 1 || ch - lane < ep.C) ep.tile_mt(tmem_base + lane_base + acc * (MT * R) + mt * R, tile, ch, mt, half, cx);
            }
            tc_fence_before();
            mbar_arrive(&tempty[acc]);
        }
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) ep.finish_mt((mg * MT + mt) * 128 + chl, mt, grp * 2 + half);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) tmem_dealloc<TCOLS>(tmem_base);
}

// =================================================================================================
//  The dW kernel:  dW[n, k] = sum over rows of Y^T[n, row] * X^T[k, row]
//  Both operands are K-major with K = rows: line = channel, 64 rows per line and per stage.  For layer 1 the
//  X side is the gathered concat tile (line = row, elements = input columns), i.e. an MN-major B operand.
//  Accumulators stay in TMEM over the CTA's whole row range; one epilogue at the end writes the partial.
// =================================================================================================
struct DwParams {
    int64_t rows;              // host value, or ...
    const int64_t *rows_dev;   // ... the device scalar of the compacted SLOTS layout (wins when non-NULL)
    int n_out;                 // Y channels (rows of dW)
    int nbl_total;             // X lines over all N groups (blockIdx.z), multiple of 16; a group handles <= 256
    int k_total;               // columns of the partial (all N groups), rounded up to a multiple of 4 (row stride)
    float *partial;            // [splits = gridDim.x][n_out][k_total]; atomic mode: ONE zeroed [n_out][k_total] all splits add to
    int atomic;
    int stages, stage_bytes;   // operand ring (set by launch_dw)
};

template <class SRC>
struct LineFillK {  // K-major X side from a feature-major source
    static constexpr bool B_MN = false;
    static constexpr bool USES_TMA = false;
    SRC src;
    static __host__ __device__ int bytes(int nb_lines) { return nb_lines * LINE_BYTES; }
    __device__ __forceinline__ void resolve(int64_t r) { src.resolve(r); }
    __device__ __forceinline__ void fill(uint8_t *B, int lt, int64_t r0, int ng, int nb_lines, const unsigned (&inf)[8])
    {
        for (int line = lt; line < nb_lines; line += NUM_LOAD) {
            const int ch = ng * 256 + line;
            uint4 v[8];
#pragma unroll
            for (int g = 0; g < 8; ++g) v[g] = src.chunk_i(ch, r0 + g * 8, inf[g]);
#pragma unroll
            for (int g = 0; g < 8; ++g) *reinterpret_cast<uint4 *>(B + line_chunk_off(line, g)) = v[g];
        }
    }
    static __device__ __forceinline__ uint64_t b_desc(uint32_t b_saddr, int ks) { return smem_desc_sw128(b_saddr + ks * 32, 16, ATOM_BYTES); }
};

// K-major X side fetched by TMA: the stored activation tensor a[c][ld] (c a multiple of 64) in 64-line boxes, then the
// 16-line box of the row-valid vector whose first line is the "ones" line (bias gradient).  No loader arithmetic.
struct TmaFill {
    static constexpr bool B_MN = false;
    static constexpr bool USES_TMA = true;
    int c;         // channels of the tensor; with the ones box: a multiple of 64 with (c % 256) + 16 <= 256
    int ones_box;  // 1: append the row-valid box at line c; 0: the tensor carries its own ones line (layer-1 operand)
    // the copies come in whole 64-line boxes: the tile must hold them even when fewer lines are used
    static __host__ __device__ int bytes(int nb_lines) { return ((nb_lines + 63) / 64) * 64 * LINE_BYTES; }
    __device__ __forceinline__ void resolve(int64_t) {}
    __device__ __forceinline__ void fill(uint8_t *, int, int64_t, int, int, const unsigned (&)[8]) {}
    // N group ng covers lines [256 ng, 256 ng + 256) of [tensor channels | ones line | zero padding]
    // lines of the X tile the copies of N group ng write (whole 64-line boxes + the 16-line ones box)
    __device__ __forceinline__ int landed_lines(int ng) const
    {
        const int ch0 = ng * 256;
        const int left = c - ch0;
        const int boxes = left <= 0 ? 0 : ((left < 256 ? left : 256) + 63) >> 6;
        const bool ones_here = ones_box && c >= ch0 && c < ch0 + 256;
        const int tensor_lines = boxes * 64;
        return ones_here ? max(tensor_lines, c - ch0 + 16) : tensor_lines;
    }
    __device__ __forceinline__ unsigned fill_tma(uint8_t *B, int64_t r0, int ng, const TmaMap *map_x, const TmaMap *map_v,
                                                 uint64_t *bar) const
    {
        const int ch0 = ng * 256;
        const int left = c - ch0;
        const int boxes = left <= 0 ? 0 : ((left < 256 ? left : 256) + 63) >> 6;
        const bool ones_here = ones_box && c >= ch0 && c < ch0 + 256;
        const unsigned bytes = (unsigned)((boxes * 64 + (ones_here ? 16 : 0)) * LINE_BYTES);
        mbar_expect_tx(bar, bytes);
        for (int blk = 0; blk < boxes; ++blk) tma_load_2d(B + blk * (64 * LINE_BYTES), map_x, (int)r0, ch0 + blk * 64, bar);
        if (ones_here) tma_load_2d(B + (c - ch0) * LINE_BYTES, map_v, (int)r0, 0, bar);
        return bytes;
    }
    static __device__ __forceinline__ uint64_t b_desc(uint32_t b_saddr, int ks) { return smem_desc_sw128(b_saddr + ks * 32, 16, ATOM_BYTES); }
};

struct LineFillGather {  // MN-major X side: [column blocks of 64][64 row lines]; thread lt: row line lt>>1, half of the chunks
    static constexpr bool B_MN = true;
    static constexpr bool USES_TMA = false;
    GatherLoaderTC g;
    static __host__ __device__ int bytes(int nb_lines) { return ((nb_lines + 63) / 64) * 64 * LINE_BYTES; }
    __device__ __forceinline__ void resolve(int64_t r) { g.resolve(r); }
    __device__ __forceinline__ void fill(uint8_t *B, int lt, int64_t r0, int ng, int nb_lines, const unsigned (&inf)[8])
    {
        const int rl = lt >> 1, half = lt & 1;
        g.set_row(r0 + rl);
        const int nblk = (nb_lines + 63) / 64;
        for (int blk = 0; blk < nblk; ++blk) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int cc = half * 4 + c;
                *reinterpret_cast<uint4 *>(B + blk * (64 * LINE_BYTES) + line_chunk_off(rl, cc)) =
                    g.chunk(ng * 256 + blk * 64 + cc * 8);
            }
        }
    }
    // K = row lines: 16 lines per step; LBO = stride between 64-column blocks, SBO = 8 lines
    static __device__ __forceinline__ uint64_t b_desc(uint32_t b_saddr, int ks)
    {
        return smem_desc_sw128(b_saddr + ks * (16 * LINE_BYTES), 64 * LINE_BYTES, ATOM_BYTES);
    }
};

template <int MTA>
struct DwPlan {
    static constexpr int A_BYTES = MTA * 128 * LINE_BYTES;
    static constexpr int MAX_STAGES = 8;
    static constexpr int SMEM_BUDGET = 222 * 1024;  // of the 227 KB a CTA may have
};

template <int MTA, class YS, class XF>
__global__ void __launch_bounds__(NT, 1) tc_dw_kernel(const DwParams p, YS ys, XF xf, const __grid_constant__ TmaMap tmap_y,
                                                       const __grid_constant__ TmaMap tmap_x, const __grid_constant__ TmaMap tmap_v)
{
    using P = DwPlan<MTA>;
    static_assert(YS::USES_TMA || YS::SCATTER, "the Y tile comes by TMA or is built by the routed-gradient fill groups");
    // the operand ring is sized at launch: stage = A tile + the X lines actually used, as many stages as fit (<= 8) --
    // with TMA-fed operands the kernel is a pure stream and lives off the bytes it keeps in flight
    const int nst = p.stages, sbytes = p.stage_bytes;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + nst * sbytes);
    uint64_t *empty = full + nst;
    uint64_t *done = empty + nst;
    uint64_t *xland = done + 1;  // per stage: the X tile's TMA copies have landed (it is converted fp16 -> bf16 in place)
    uint32_t *tmem_holder = reinterpret_cast<uint32_t *>(xland + nst);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int split = blockIdx.x, mg = blockIdx.y, ng = blockIdx.z;
    constexpr int TCOLS = MTA * 256;
    const int64_t rows = p.rows_dev ? *p.rows_dev : p.rows;
    ys.resolve(rows);
    xf.resolve(rows);
    const int64_t chunks = (rows + 63) / 64;
    const int64_t cps = (chunks + gridDim.x - 1) / gridDim.x;
    const int64_t c_beg = (int64_t)split * cps;
    const int64_t c_end = min(chunks, c_beg + cps);
    const int64_t nchunks = c_end > c_beg ? c_end - c_beg : 0;
    const int nb_lines = min(256, p.nbl_total - ng * 256);

    if (tid == 0) {
        for (int s = 0; s < nst; ++s) {
            mbar_init(&full[s], YS::SCATTER ? 2 * NUM_LOAD : NUM_LOAD);   // converter group (+ fill group of a routed Y side)
            mbar_init(&empty[s], 1);
            mbar_init(&xland[s], 1);
        }
        mbar_init(done, 1);
        fence_barrier_init();
    }
    if (warp == MMA_WARP) tmem_alloc<TCOLS>(tmem_holder);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    // Kernels whose operands all come through TMA and whose warps 0-7 have nothing else to do get a DEDICATED producer thread
    // (warp 4, lane 0): it refills a stage the moment the MMA releases it instead of when a converter thread next comes
    // round its loop.  Routed kernels (warps 0-7 build the Y tile) keep the issue in the converter groups.
    constexpr bool ANY_TMA = YS::USES_TMA || XF::USES_TMA;
    constexpr bool DEDICATED = ANY_TMA && !YS::SCATTER;
    // TMA copies of chunk i (one thread): the Y tile completes on full[s] directly; the X tile lands as fp16 and completes
    // on xland[s], because the group converts it to bf16 before the MMA may read it.  The copies are issued up to
    // AHEAD chunks of this group ahead of the conversion, so the ring stays as deep as before the conversion existed
    // (these kernels are pure streams: they live off the bytes in flight).
    auto issue = [&](int64_t i) {
        const int s = (int)(i % nst);
        const uint32_t ph = (uint32_t)(i / nst) & 1u;
        uint8_t *A = smem + s * sbytes;
        uint8_t *B = A + P::A_BYTES;
        const int64_t r0 = (c_beg + i) * 64;
        mbar_wait(&empty[s], ph ^ 1u);
        if constexpr (YS::USES_TMA) {  // MTA*128 lines x 64 rows straight from the feature-major tensor, 64 lines per copy
            mbar_expect_tx(&full[s], P::A_BYTES);
#pragma unroll
            for (int m = 0; m < MTA * 2; ++m)
                tma_load_2d(A + m * (64 * LINE_BYTES), &tmap_y, (int)r0, mg * (MTA * 128) + m * 64, &full[s]);
        }
        if constexpr (XF::USES_TMA) {
            xf.fill_tma(B, r0, ng, &tmap_x, &tmap_v, &xland[s]);
            mbar_arrive(&xland[s]);
        }
    };
    // converter / loader groups: warps 8-11 and 12-15; with a dedicated producer also warps 0-3 (idle until the final drain)
    constexpr int NG = DEDICATED ? LOAD_GROUPS + 1 : LOAD_GROUPS;
    if ((warp >= NUM_EPI / 32 && warp < MMA_WARP) || (DEDICATED && warp < 4)) {
        const int grp = warp < 4 ? LOAD_GROUPS : (tid - NUM_EPI) / NUM_LOAD;
        const int lt = warp < 4 ? tid : (tid - NUM_EPI) % NUM_LOAD;
        // group descriptors of the 64 rows of a chunk (unused, and dropped by the compiler, for TMA-fed operands); the ones
        // of the group's NEXT chunk are requested before the current chunk is built
        auto load_inf = [&](unsigned (&inf)[8], int64_t r0) {
            if (ys.rm.seg_mode) {
#pragma unroll
                for (int g = 0; g < 8; ++g) inf[g] = ys.rm.info(r0 + g * 8);
            } else {
#pragma unroll
                for (int g = 0; g < 8; ++g) inf[g] = ys.rm.info_slots(r0 + g * 8);
            }
        };
        unsigned inf[8], infn[8];
        if (grp < nchunks) load_inf(inf, (c_beg + grp) * 64);
        const int ahead = nst / NG > 1 ? nst / NG : 1;  // chunks of this group in flight
        int64_t iss = grp;
        for (int64_t i = grp; i < nchunks; i += NG) {
            const int s = (int)(i % nst);
            const uint32_t ph = (uint32_t)(i / nst) & 1u;
            uint8_t *A = smem + s * sbytes;
            uint8_t *B = A + P::A_BYTES;
            const int64_t r0 = (c_beg + i) * 64;
            if (i + NG < nchunks) load_inf(infn, (c_beg + i + NG) * 64);
            if constexpr (ANY_TMA && !DEDICATED) {
                // a wait in issue() depends on chunks < iss - nst + 1 <= i only, i.e. on work this group has already done
                if (lt == 0)
                    for (; iss < nchunks && iss < i + (int64_t)ahead * NG; iss += NG) issue(iss);
            }
            // (a routed Y tile is built by the fill groups, warps 0-7, below)
            if constexpr (XF::USES_TMA) {
                // the stored activations are fp16, the gradients on the Y side bf16: the group converts the landed X tile
                // to bf16 in place (16-byte chunks, element-wise: the swizzle is untouched).  Every thread first makes sure
                // the stage's PREVIOUS use has been consumed (with an odd number of stages the two groups alternate on a
                // stage, and a parity wait on xland alone could be satisfied by the use before the previous one)
                mbar_wait(&empty[s], ph ^ 1u);
                mbar_wait(&xland[s], ph);
                const int nchunk16 = xf.landed_lines(ng) * 8;
                for (int c = lt; c < nchunk16; c += NUM_LOAD) {
                    uint4 *q = reinterpret_cast<uint4 *>(B) + c;
                    *q = f16_to_bf16_chunk(*q);
                }
            } else {
                mbar_wait(&empty[s], ph ^ 1u);
                xf.fill(B, lt, r0, ng, nb_lines, inf);
            }
            fence_proxy_async_smem();
            mbar_arrive(&full[s]);
#pragma unroll
            for (int g = 0; g < 8; ++g) inf[g] = infn[g];
        }
    } else if (warp == MMA_WARP) {
        if (lane == 0 && nchunks > 0) {
            // both operands are bf16 at MMA time: kind::f16 wants ONE format for A and B (a bf16 x fp16 instruction is an
            // illegal instruction on sm_100a -- measured), so the fp16 activations are converted on their way in
            const uint32_t idesc = idesc_bf16(128, nb_lines, false, XF::B_MN);
            for (int64_t i = 0; i < nchunks; ++i) {
                const int s = (int)(i % nst);
                const uint32_t ph = (uint32_t)(i / nst) & 1u;
                mbar_wait(&full[s], ph);
                tc_fence_after();
                const uint32_t a_s = smem_u32(smem + s * sbytes);
                const uint32_t b_s = a_s + P::A_BYTES;
#pragma unroll
                for (int mt = 0; mt < MTA; ++mt) {
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t ad = smem_desc_sw128(a_s + mt * (128 * LINE_BYTES) + ks * 32, 16, ATOM_BYTES);
                        const uint64_t bd = XF::b_desc(b_s, ks);
                        umma_bf16(tmem_base + mt * 256, ad, bd, idesc, (i | ks) != 0);
                    }
                }
                umma_commit(&empty[s]);
            }
            umma_commit(done);
        }
    } else {
        if constexpr (DEDICATED) {
            if (warp == 4 && lane == 0)
                for (int64_t i = 0; i < nchunks; ++i) issue(i);
        }
        if constexpr (YS::SCATTER) {
            // Routed-gradient Y side: warps 0-7 (idle until the final drain otherwise) form two FILL groups of 128 threads that
            // take alternate chunks; the loader groups above only convert the X tile.  A group zeroes the Y tile, meets at its
            // named barrier and drops quads (see RouteSource).  Work item k of thread lt: channel quad (lt + 128 k) % NQ, row
            // group (lt + 128 k) / NQ.  A software pipeline per thread: descriptors three chunks ahead, the rows of the chunk
            // two ahead pulled into L2, (arg, dout) quads one chunk ahead, the stores of the current chunk.
            const int grp = tid / NUM_LOAD;
            const int lt = tid % NUM_LOAD;
            constexpr int NQ = MTA * 32, NI = MTA * 2;
            RouteSource::Quad qd[NI];
            // descriptors: qi = this chunk (normalised); r1 / r2 / r3 = the group's next three chunks as RAW table words + a
            // "past the end" mask (normalising a word where it is requested would wait for the load on the spot)
            unsigned qi[NI], r1[NI], r2[NI], r3[NI], d1 = 0u, d2 = 0u, d3 = 0u;
            auto q_fetch = [&](unsigned (&w)[NI], unsigned &dead, int64_t i) {
                dead = 0u;
#pragma unroll
                for (int k = 0; k < NI; ++k) {
                    if (i < nchunks) {
                        const int64_t r8 = (c_beg + i) * 64 + ((lt + NUM_LOAD * k) / NQ) * 8;
                        w[k] = __ldg(ys.rm.rgrp + (r8 >> 3));
                        dead |= (r8 >= ys.rm.rows ? 1u : 0u) << k;
                    } else {
                        w[k] = GI_NONE;
                        dead |= 1u << k;
                    }
                }
            };
            auto q_norm = [&](const unsigned (&w)[NI], unsigned dead) {
#pragma unroll
                for (int k = 0; k < NI; ++k) qi[k] = (((dead >> k) & 1u) || gi_none(w[k])) ? GI_NONE : w[k];
            };
            auto q_load = [&]() {
#pragma unroll
                for (int k = 0; k < NI; ++k) ys.load_quad(qi[k], mg * (MTA * 128) + ((lt + NUM_LOAD * k) % NQ) * 4, qd[k]);
            };
            // every (arg, dout) row is read exactly once: a compulsory DRAM miss the one-chunk-ahead register prefetch cannot
            // cover; one thread per 128 bytes pulls them into L2 two chunks ahead
            auto q_prefetch = [&](const unsigned (&w)[NI], unsigned dead) {
#pragma unroll
                for (int k = 0; k < NI; ++k) {
                    const int q = (lt + NUM_LOAD * k) % NQ;
                    const int ch4 = mg * (MTA * 128) + q * 4;
                    if ((q & 7) != 0 || ((dead >> k) & 1u) || gi_none(w[k]) || gi_nv(w[k]) == 0 || gi_slot0(w[k]) != 0 || ch4 >= ys.C) continue;
                    const int64_t idx = (int64_t)gi_seg(w[k]) * ys.C + ch4;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(ys.arg + idx));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(ys.dout + idx));
                }
            };
#pragma unroll
            for (int k = 0; k < NI; ++k) qi[k] = r1[k] = r2[k] = r3[k] = GI_NONE;
            if (grp < nchunks) {
                q_fetch(r1, d1, grp);
                q_norm(r1, d1);
                q_load();
                q_fetch(r1, d1, grp + LOAD_GROUPS);
                q_fetch(r2, d2, grp + 2 * LOAD_GROUPS);
            }
            for (int64_t i = grp; i < nchunks; i += LOAD_GROUPS) {
                const int s = (int)(i % nst);
                const uint32_t ph = (uint32_t)(i / nst) & 1u;
                uint8_t *A = smem + s * sbytes;
                q_fetch(r3, d3, i + 3 * LOAD_GROUPS);
                q_prefetch(r2, d2);
                mbar_wait(&empty[s], ph ^ 1u);
                RouteSource::zero_tile(smem_u32(A), P::A_BYTES, lt);
                RouteSource::group_barrier(1 + grp);
#pragma unroll
                for (int k = 0; k < NI; ++k) {
                    const int l0 = ((lt + NUM_LOAD * k) % NQ) * 4, g = (lt + NUM_LOAD * k) / NQ;
                    const int ch4 = mg * (MTA * 128) + l0;
                    ys.store_quad(qd[k], ys.starts(qi[k], ch4), ch4, g, smem_u32(A), l0);
                }
                fence_proxy_async_smem();
                mbar_arrive(&full[s]);
                // the quads of this group's next chunk travel while the MMA and the other group work
                if (i + LOAD_GROUPS < nchunks) {
                    q_norm(r1, d1);
                    q_load();
                }
#pragma unroll
                for (int k = 0; k < NI; ++k) {
                    r1[k] = r2[k];
                    r2[k] = r3[k];
                }
                d1 = d2, d2 = d3;
            }
        }
    }
    if (warp < 4) {   // the final drain of the accumulators
        {
        if (nchunks > 0) {
            mbar_wait(done, 0);
            tc_fence_after();
        }
        const uint32_t lane_base = ((uint32_t)(warp * 32)) << 16;
#pragma unroll
        for (int mt = 0; mt < MTA; ++mt) {
            const int ch = (mg * MTA + mt) * 128 + tid;
            float *dst = p.partial + ((int64_t)(p.atomic ? 0 : split) * p.n_out + ch) * p.k_total + ng * 256;
            if (p.atomic && nchunks == 0) continue;  // nothing to add
            for (int cc = 0; cc * 32 < nb_lines; ++cc) {
                float v[32];
                if (nchunks > 0) {
                    tmem_ld32(tmem_base + lane_base + mt * 256 + cc * 32, v);
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = 0.f;
                }
                if (ch < p.n_out) {  // k_total (the partial's row stride) is a multiple of 4: 16-byte stores
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const int col = cc * 32 + q * 4;
                        if (col < nb_lines && ng * 256 + col < p.k_total) {
                            if (p.atomic)
                                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + col), "f"(v[4 * q]),
                                             "f"(v[4 * q + 1]), "f"(v[4 * q + 2]), "f"(v[4 * q + 3])
                                             : "memory");
                            else
                                *reinterpret_cast<float4 *>(dst + col) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
                        }
                    }
                }
            }
        }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) tmem_dealloc<TCOLS>(tmem_base);
}

// =================================================================================================
//  small kernels
// =================================================================================================
// bf16 operand image of a weight matrix: element (m, k) = w[m*sm + col(k)*sk] for m < M, k < Kimg (col(k) is the
// identity, or InCols::src_col for the layer-1 operand), else 0.
// Layout: [m_group][k_chunk][MT*128 lines][128 B] with the 128B swizzle applied per line.
struct PackJob {
    const float *w;
    int M, Kimg;
    int64_t sm, sk;
    int use_map;
    InCols cols;
    int MT, num_mg, num_kc;
    uint8_t *img;
    int fmt;  // FMT_F16 (forward weights) / FMT_BF16 (transposed weights that meet gradients)
    // 64-row matrices only: lines 64..127 of the image repeat rows 0..63 instead of holding zeros, so the accumulator has
    // every channel on TWO TMEM lanes (c and 64 + c) and all four lane quadrants' warps can drain it (sa_chain.cuh)
    int dup64;
};
struct PackJobs {
    PackJob j[3];
};
// blockIdx.y selects the matrix: all weight images of a forward / backward call in ONE launch
__global__ void pack_weights_kernel(const PackJobs jobs)
{
    const PackJob &jb = jobs.j[blockIdx.y];
    const int lines = jb.MT * 128;
    const int64_t total = (int64_t)jb.num_mg * jb.num_kc * lines * 8;  // one thread per 16-byte chunk
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i & 7);
        const int64_t t = i >> 3;
        const int line = (int)(t % lines);
        const int64_t t2 = t / lines;
        const int kc = (int)(t2 % jb.num_kc);
        const int mgi = (int)(t2 / jb.num_kc);
        int m = mgi * lines + line;
        if (jb.dup64 && m >= 64 && m < 128) m -= 64;
        float f[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int k = kc * KC + c * 8 + e;
            int col = k < jb.Kimg ? k : -1;
            if (jb.use_map && col >= 0) col = jb.cols.src_col(k);
            f[e] = (m < jb.M && col >= 0) ? jb.w[(int64_t)m * jb.sm + (int64_t)col * jb.sk] : 0.f;
        }
        uint8_t *dst = jb.img + (((int64_t)mgi * jb.num_kc + kc) * lines) * LINE_BYTES + line_chunk_off(line, c);
        *reinterpret_cast<uint4 *>(dst) = jb.fmt == FMT_F16 ? pack8h(f) : pack8(f);
    }
}

static inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

struct Packed {
    uint8_t *img;
    int MT, num_mg, num_kc;
    int64_t bytes;
    int fmt;
};
static Packed plan_pack(int M, int Kimg, int fmt)
{
    Packed p;
    p.fmt = fmt;
    const int mpad = (int)align_up(M, 128);
    p.MT = mpad >= 256 ? 2 : 1;
    p.num_mg = (mpad + p.MT * 128 - 1) / (p.MT * 128);
    p.num_kc = (Kimg + KC - 1) / KC;
    p.bytes = (int64_t)p.num_mg * p.num_kc * p.MT * 128 * LINE_BYTES;
    p.img = nullptr;
    return p;
}
static PackJob pack_job(const float *w, int M, int Kimg, int64_t sm, int64_t sk, const InCols *map, const Packed &p)
{
    PackJob j = {w, M, Kimg, sm, sk, map ? 1 : 0, map ? *map : InCols{0, 0}, p.MT, p.num_mg, p.num_kc, p.img, p.fmt};
    return j;
}
static void launch_packs(const PackJob *jobs, int n, cudaStream_t st)
{
    if (n <= 0) return;
    PackJobs pj;
    int64_t mx = 0;
    for (int i = 0; i < 3; ++i) {
        pj.j[i] = jobs[i < n ? i : 0];
        const int64_t tot = (int64_t)pj.j[i].num_mg * pj.j[i].num_kc * pj.j[i].MT * 128 * 8;
        mx = tot > mx ? tot : mx;
    }
    int64_t bx = (mx + 255) / 256;
    if (bx > 592) bx = 592;  // grid-stride beyond 4 blocks per SM
    pack_weights_kernel<<<dim3((unsigned)bx, (unsigned)n), 256, 0, st>>>(pj);
    note_launch();
}
static void launch_pack(const float *w, int M, int Kimg, int64_t sm, int64_t sk, const InCols *map, const Packed &p,
                        cudaStream_t st)
{
    const PackJob j = pack_job(w, M, Kimg, sm, sk, map, p);
    launch_packs(&j, 1, st);
}

}  // namespace tc
}  // namespace b2pn
#include "sa_chain.cuh"
namespace b2pn {
namespace tc {

// SM count of the current device
static int device_sms()
{
    static int sms_of[64] = {};  // per device; a racing first call writes the same value twice
    int dev = 0;
    cudaGetDevice(&dev);
    int sms = (dev >= 0 && dev < 64) ? sms_of[dev] : 0;
    if (sms == 0) {
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
        if (dev >= 0 && dev < 64) sms_of[dev] = sms;
    }
    return sms;
}

// CTAs the persistent kernels of one call may take: one per SM, or b2pn_sa_args::sm_limit, which leaves SMs free for
// kernels of a concurrent stream (these kernels take one CTA per SM and stride over tiles by gridDim.x, so a CTA that
// cannot become resident would double their time)
static int cta_budget(const b2pn_sa_args &a)
{
    const int sms = device_sms();
    return (a.sm_limit > 0 && a.sm_limit < sms) ? a.sm_limit : sms;
}

// grid.x of a rows-GEMM launch (the per-CTA statistics partials are indexed by blockIdx.x)
static int grid_x_for(const Packed &pk, int64_t tiles, int ctas)
{
    int gx = ctas / pk.num_mg;
    if (gx < 1) gx = 1;
    if ((int64_t)gx > tiles) gx = (int)tiles;
    return gx;
}

// rows of a launch: an upper bound known on the host (sizes the grid) and, for the compacted SLOTS layout, the
// device scalar holding the real count; and the CTAs the launch may take (cta_budget)
struct RowsArg {
    int64_t cap;
    const int64_t *dev;
    int ctas;
    int64_t tiles() const { return (cap + R - 1) / R; }
};

static const TmaMap kNoMap = {};

template <int MT, class BL, class EP>
static int launch_gemm(const Packed &pk, const RowsArg &ra, const BL &bl, const EP &ep, cudaStream_t st,
                       const TmaMap &map = kNoMap, const TmaMap &e0 = kNoMap, const TmaMap &e1 = kNoMap)
{
    using P = SmemPlan<MT, EP::STAGED, BL::WIDE>;
    auto kern = tc_rows_gemm_kernel<MT, BL, EP>;
    static SmemAttrSlot slot = {};
    cudaError_t e = ensure_dynamic_smem(kern, P::TOTAL, slot);
    if (e != cudaSuccess) return (int)e;
    GemmParams gp = {pk.img, pk.fmt, pk.fmt, pk.num_kc, ra.cap, ra.dev};
    dim3 grid((unsigned)grid_x_for(pk, ra.tiles(), ra.ctas), (unsigned)pk.num_mg);
    kern<<<grid, gemm_threads<BL>(), P::TOTAL, st>>>(gp, bl, ep, map, e0, e1);
    note_launch();
    e = cudaPeekAtLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

template <class BL, class EP1, class EP2>
static int launch_by_mt(const Packed &pk, const RowsArg &ra, const BL &bl, const EP1 &e1, const EP2 &e2, cudaStream_t st,
                        const TmaMap &map = kNoMap, const TmaMap &m0 = kNoMap, const TmaMap &m1 = kNoMap)
{
    return pk.MT == 1 ? launch_gemm<1>(pk, ra, bl, e1, st, map, m0, m1) : launch_gemm<2>(pk, ra, bl, e2, st, map, m0, m1);
}

// number of rows the BatchNorm statistics run over: a host constant (CLOUDS) or the edge count b2pn_pack_rows left next
// to the row count (SLOTS: num_rows[1])
struct CountArg {
    const int64_t *dev;
    double host;
    __device__ __forceinline__ double get() const { return dev ? (double)*dev : host; }
};

// partial[g][2][cpad]: per-CTA sums of the bias-free accumulators over ALL rows (invalid rows are exact zeros):
//   mean(h) = S/E + bias,  var(h) = Q/E - (S/E)^2.   bn = [mean, rstd, scale, shift] x cmax
__device__ __forceinline__ void warp_sum_partials(const double *partial, int gx, int cpad, int c, double &S, double &Q)
{
    const int lane = threadIdx.x & 31;
    double s = 0.0, q = 0.0;
    {
        // all of a lane's partials (<= 4 slots x MAX_GX CTAs / 32 lanes) are requested before the first one is used:
        // one L2 round trip; fixed summation order
        constexpr int PER = (4 * 160 + 31) / 32;
        double sv[PER], qv[PER];
#pragma unroll
        for (int u = 0; u < PER; ++u) {
            const int g = lane + 32 * u;
            const bool in = g < gx;
            const int64_t o = in ? (int64_t)g * 2 * cpad + c : c;
            sv[u] = partial[o];
            qv[u] = partial[o + cpad];
            if (!in) sv[u] = qv[u] = 0.0;
        }
#pragma unroll
        for (int u = 0; u < PER; ++u) {
            s += sv[u];
            q += qv[u];
        }
    }
    // fixed-order butterfly: deterministic
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    S = s;
    Q = q;
}

// one warp per channel
__global__ void bn_fwd_finalize_tc_kernel(const double *partial, int gx, int C, int cpad, const CountArg count, int training,
                                          const float *bias, const float *gamma, const float *beta, float *running_mean,
                                          float *running_var, int64_t *nbt, float eps, float momentum, float *bn, int cmax)
{
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (c >= C) return;
    double mean, var;
    if (training) {
        double S, Q;
        warp_sum_partials(partial, gx, cpad, c, S, Q);
        const double E = count.get();
        const double ma = E > 0 ? S / E : 0.0;
        mean = ma + (double)bias[c];
        var = E > 0 ? Q / E - ma * ma : 0.0;
        if (var < 0.0) var = 0.0;
        if ((threadIdx.x & 31) == 0) {
            const double unbiased = E > 1.0 ? var * E / (E - 1.0) : var;
            running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * mean);
            running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unbiased);
            if (c == 0 && nbt) *nbt += 1;
        }
    } else {
        mean = running_mean[c];
        var = running_var[c];
    }
    if ((threadIdx.x & 31) == 0) {
        const double rstd = 1.0 / sqrt(var + (double)eps);
        const double scale = (double)gamma[c] * rstd;
        bn[c] = (float)mean;
        bn[cmax + c] = (float)rstd;
        bn[2 * cmax + c] = (float)scale;
        bn[3 * cmax + c] = (float)((double)beta[c] - mean * scale);
    }
}

// S1 = sum dz, S2 = sum dz*zhat -> dbeta, dgamma, and the per-channel means the BN backward needs
__global__ void bn_bwd_finalize_tc_kernel(const double *partial, int gx, int C, int cpad, const CountArg count, int training,
                                          float *grad_gamma, float *grad_beta, float *sbar)
{
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (c >= C) return;
    double S, Q;
    warp_sum_partials(partial, gx, cpad, c, S, Q);
    if ((threadIdx.x & 31) == 0) {
        const double E = count.get();
        if (grad_beta) grad_beta[c] = (float)S;
        if (grad_gamma) grad_gamma[c] = (float)Q;
        sbar[c] = (training && E > 0) ? (float)(S / E) : 0.f;
        sbar[C + c] = (training && E > 0) ? (float)(Q / E) : 0.f;
    }
}

// Routed gradient of the global max pool as a dense feature-major bf16 tensor (CLOUDS levels):
//   dh3[ch][row] = dout[b][ch] if row is the arg-max source row of (cloud b = batch[row], ch), else 0.
// Written once so that both consumers (dX of the last layer and dW3) take it through the TMA unit.  (SLOTS levels build
// their routed tiles in the loaders instead: RouteSource.)  Thread = (channel, 8-row group), groups fastest: 16-byte stores
// coalesce along the rows, the (arg, dout) reads stay L2-resident.
__global__ void route_grad_clouds_tc_kernel(RowMapTC rm, const int64_t *rows_dev, const float *dout, const int32_t *arg, int C,
                                            int64_t ld, __nv_bfloat16 *dh)
{
    if (rows_dev) rm.rows = *rows_dev;
    const int64_t groups = (rm.rows + 127) / 128 * 16;  // whole tiles
    const int64_t total = groups * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int ch = (int)(i / groups);
        const int64_t g = i - (int64_t)ch * groups;
        const unsigned inf = rm.info(g * 8);
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        float f[8];
        bool any = false;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int64_t row = g * 8 + e;
            f[e] = 0.f;
            if (e < gi_nv(inf)) {
                const int64_t sg = __ldg(rm.batch + row);
                if ((int64_t)__ldg(arg + sg * C + ch) == row) {
                    f[e] = __ldg(dout + sg * C + ch);
                    any = true;
                }
            }
        }
        if (any) v = pack8(f);
        *reinterpret_cast<uint4 *>(dh + (int64_t)ch * ld + g * 8) = v;
    }
}

// dh = scale * (dz - mean(dz) - zhat * mean(dz*zhat)) on valid rows, 0 elsewhere; in place, feature-major bf16
__global__ void bn_bwd_apply_tc_kernel(RowMapTC rm, const int64_t *rows_dev, __nv_bfloat16 *dz, const __nv_bfloat16 *z, int C,
                                       int64_t ld, const float *scale, const float *sbar)
{
    if (rows_dev) rm.rows = *rows_dev;
    const int64_t groups = (rm.rows + 127) / 128 * 16;  // whole tiles: the pad rows of the last tile are zeroed too
    const int64_t total = groups * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int ch = (int)(i / groups);
        const int64_t r8 = (i - (int64_t)ch * groups) * 8;
        const int nv = rm.valid8(r8);
        uint4 *p = reinterpret_cast<uint4 *>(dz + (int64_t)ch * ld + r8);
        if (nv == 0) {
            *p = make_uint4(0u, 0u, 0u, 0u);
            continue;
        }
        float d[8], zf[8];
        unpack8(*p, d);
        unpack8h(__ldg(reinterpret_cast<const uint4 *>(z + (int64_t)ch * ld + r8)), zf);
        const float sc = scale[ch];
        const float s1 = sbar[ch], s2 = sbar[C + ch];
#pragma unroll
        for (int e = 0; e < 8; ++e) d[e] = e < nv ? sc * (d[e] - s1 - zf[e] * s2) : 0.f;
        *p = pack8(d);
    }
}

// dW = sum over the split partials; image columns that share a weight column (hi/lo parts) are added up;
// the "ones" image column is the bias gradient.  blockIdx.y selects the layer: the three weight gradients of a level are
// reduced by ONE launch at the end of its backward pass (each is a string of dependent L2 round trips, not bandwidth).
struct DwReduceJob {
    const float *partial;
    int splits, n_out, k_total, use_map;
    InCols cols;
    int k_true, ones_idx;
    float *grad_w, *grad_b;
};
struct DwReduceJobs {
    DwReduceJob j[3];
};
// (a) one thread per output element, 16 loads in flight: for large outputs / few splits (bandwidth bound)
__global__ void dw_reduce_flat_tc_kernel(const DwReduceJobs jobs)
{
    const DwReduceJob &jb = jobs.j[blockIdx.y];
    const int k_true = jb.k_true, k_total = jb.k_total, n_out = jb.n_out, splits = jb.splits;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per output element (coalesced)
    if (i >= (int64_t)n_out * (k_true + 1)) return;
    const int n = (int)(i / (k_true + 1));
    const int k = (int)(i - (int64_t)n * (k_true + 1));
    int c0 = -1, c1 = -1;
    if (k == k_true) {
        c0 = jb.ones_idx;
    } else if (!jb.use_map) {
        c0 = k;
    } else {
        const int nx = jb.cols.nx();
        if (k < jb.cols.c_in) {
            c0 = k;
            c1 = jb.cols.x_f32 ? k + jb.cols.c_in : -1;
        } else {
            c0 = nx + (k - jb.cols.c_in);
            c1 = c0 + 3;
        }
    }
    const int64_t stride = (int64_t)n_out * k_total;
    const float *base = jb.partial + (int64_t)n * k_total;
    constexpr int U = 16;  // independent chains: keep 16 loads in flight; fixed order
    double acc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) acc[u] = 0.0;
    int p = 0;
    for (; p + U <= splits; p += U) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const float *row = base + (int64_t)(p + u) * stride;
            float v = row[c0];
            if (c1 >= 0) v += row[c1];
            acc[u] += (double)v;
        }
    }
    for (; p < splits; ++p) {
        const float *row = base + (int64_t)p * stride;
        acc[0] += (double)row[c0];
        if (c1 >= 0) acc[0] += (double)row[c1];
    }
#pragma unroll
    for (int w = U / 2; w > 0; w >>= 1)
#pragma unroll
        for (int u = 0; u < w; ++u) acc[u] += acc[u + w];
    const double sum = acc[0];
    if (k == k_true) {
        if (jb.grad_b) jb.grad_b[n] = (float)sum;
    } else if (jb.grad_w) {
        jb.grad_w[(int64_t)n * k_true + k] = (float)sum;
    }
}

// (b) eight warps per 32 output elements: for small outputs reduced over many splits (latency bound)
constexpr int DWR_WARPS = 8;
constexpr int DWR_MAX_SPLITS = 160;  // >= the SM count (plan_dw never splits further)
__global__ void __launch_bounds__(32 * DWR_WARPS) dw_reduce_tc_kernel(const DwReduceJobs jobs)
{
    const DwReduceJob &jb = jobs.j[blockIdx.y];
    const int k_true = jb.k_true, k_total = jb.k_total, n_out = jb.n_out, splits = jb.splits;
    const int w = threadIdx.y;                                         // blockDim = (32, DWR_WARPS)
    const int64_t i = (int64_t)blockIdx.x * 32 + threadIdx.x;           // 32 output elements per block (coalesced)
    const bool live = i < (int64_t)n_out * (k_true + 1);
    const int n = live ? (int)(i / (k_true + 1)) : 0;
    const int k = live ? (int)(i - (int64_t)n * (k_true + 1)) : 0;
    int c0 = 0, c1 = -1;
    if (k == k_true) {
        c0 = jb.ones_idx;
    } else if (!jb.use_map) {
        c0 = k;
    } else {
        const int nx = jb.cols.nx();
        if (k < jb.cols.c_in) {
            c0 = k;
            c1 = jb.cols.x_f32 ? k + jb.cols.c_in : -1;
        } else {
            c0 = nx + (k - jb.cols.c_in);
            c1 = c0 + 3;
        }
    }
    const int64_t stride = (int64_t)n_out * k_total;
    const float *base = jb.partial + (int64_t)n * k_total;
    // warp w of the block takes the splits p = w, w + 8, ...: all of a thread's loads are in flight together (one L2
    // round trip instead of splits / 16 dependent ones), 128-byte coalesced per split; fixed summation order
    constexpr int PER = (DWR_MAX_SPLITS + DWR_WARPS - 1) / DWR_WARPS;
    float v[PER];
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int p = w + u * DWR_WARPS;
        v[u] = 0.f;
        if (live && p < splits) {
            const float *row = base + (int64_t)p * stride;
            v[u] = row[c0];
            if (c1 >= 0) v[u] += row[c1];
        }
    }
    double acc = 0.0;
#pragma unroll
    for (int u = 0; u < PER; ++u) acc += (double)v[u];
    __shared__ double part[DWR_WARPS][32];
    part[w][threadIdx.x] = acc;
    __syncthreads();
    if (w != 0 || !live) return;
    double sum = 0.0;
#pragma unroll
    for (int q = 0; q < DWR_WARPS; ++q) sum += part[q][threadIdx.x];
    if (k == k_true) {
        if (jb.grad_b) jb.grad_b[n] = (float)sum;
    } else if (jb.grad_w) {
        jb.grad_w[(int64_t)n * k_true + k] = (float)sum;
    }
}

__global__ void unpack_keys_tc_kernel(const unsigned long long *keys, float *out, int32_t *arg, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = keys[i];
    if (k == 0ull) {
        out[i] = 0.f;
        arg[i] = -1;
    } else {
        const unsigned o = (unsigned)(k >> 32);
        out[i] = __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
        arg[i] = (int32_t)(0xffffffffu - (unsigned)(k & 0xffffffffu));
    }
}

// -------------------------------------------------------------------------------------------------
//  self-test: out[m][row] = sum_k w[m][k] * b(row, k) with b given row-major [rows][k] bf16 (mode 0, K-major
//  B tiles through the gather loader) or feature-major [k][ld] bf16 (mode 1, MN-major B tiles)
// -------------------------------------------------------------------------------------------------
int tc_gemm_selftest(const float *w, int m_out, int k, const void *b, int mode, int64_t rows, int64_t ld, const float *zeros3,
                     float *out, int64_t ld_out, void *workspace, int64_t workspace_bytes, cudaStream_t st)
{
    if (!w || !b || !out || !workspace || !zeros3 || m_out <= 0 || k <= 0 || rows <= 0) return B2PN_EINVAL;
    // fp16 weights x fp16 operand: the forward configuration.  (A bf16 x fp16 kind::f16 instruction is an ILLEGAL
    // INSTRUCTION on sm_100a -- measured in round 2 -- which is why the dW kernel converts its fp16 X tiles to bf16.)
    if (mode < 0 || mode > 2) return B2PN_EINVAL;
    Packed pk = plan_pack(m_out, k, FMT_F16);
    if (workspace_bytes < pk.bytes + 1024) return B2PN_EINVAL;
    pk.img = (uint8_t *)align_up((int64_t)(uintptr_t)workspace, 1024);
    launch_pack(w, m_out, k, k, 1, nullptr, pk, st);
    const RowsArg ra = {rows, nullptr, device_sms()};
    RowMapTC rm = {B2PN_SEG_CLOUDS, nullptr, nullptr, nullptr, nullptr, rows, 0};
    StoreF32Ep ep = {out, m_out, ld_out};
    if (mode == 0) {
        // all k columns are bf16 features (c_in = k); the appended dpos columns multiply zero weights
        GatherLoaderTC gl = {rm, b, InCols{k, 0}, zeros3, nullptr, -1, FMT_F16};
        return launch_by_mt(pk, ra, gl, ep, ep, st);
    }
    if (mode == 2) {  // the same feature-major operand through the TMA unit
        TmaMap map;
        const int rc = make_tma_feature_major(&map, b, k, ld);
        if (rc) return rc;
        TmaFeatLoader tl;
        return launch_by_mt(pk, ra, tl, ep, ep, st, map);
    }
    FeatLoaderTC<FeatSource<0>> fl = {{rm, (const __nv_bfloat16 *)b, k, ld, 0, -1, nullptr, nullptr, FMT_F16}};
    return launch_by_mt(pk, ra, fl, ep, ep, st);
}

// =================================================================================================
//  host orchestration
// =================================================================================================
struct WsTC {
    char *base;
    int64_t off;
    explicit WsTC(void *p) : base((char *)p), off(0)
    {
        if (base) off = align_up((int64_t)(uintptr_t)base, 1024) - (int64_t)(uintptr_t)base;
    }
    template <class T>
    T *take(int64_t n)
    {
        T *r = base ? (T *)(base + off) : nullptr;
        off = align_up(off + n * (int64_t)sizeof(T), 1024);
        return r;
    }
};

struct ShapesTC {
    int64_t rows, tiles, ld;
    int c0, c1, c2, c3, cmax, cpad, k1;
    InCols cols;
    // launch options of this call
    int ctas;            // cta_budget(): grid bound of the persistent kernels
    // b2pn_sa_args::deterministic.  false: the row splits of a dW GEMM add their partials into one zeroed buffer with
    // red.global.add.v4.f32 (no partial tensor, the reduction kernel only maps columns); true: per-split partials summed
    // in a fixed order, and the grad_x scatter of SLOTS levels accumulated in fixed point (bit-reproducible)
    bool deterministic;
};
static ShapesTC shapes_tc(const b2pn_sa_args &a)
{
    ShapesTC s;
    // SLOTS: capacity of the compacted row layout (upper bound; the real count lives in *a.num_rows)
    s.rows = a.seg_mode == B2PN_SEG_CLOUDS ? a.n_src : a.row_capacity;
    s.tiles = (s.rows + R - 1) / R;
    s.ld = s.tiles * R;
    s.c0 = a.mlp.c[0];
    s.c1 = a.mlp.c[1];
    s.c2 = a.mlp.c[2];
    s.c3 = a.mlp.c[3];
    s.cmax = s.c1 > s.c2 ? s.c1 : s.c2;
    s.cols = InCols{a.c_in, a.x_dtype == B2PN_X_F32 ? 1 : 0};
    s.k1 = s.cols.k_img();
    int mx = s.cmax > s.c3 ? s.cmax : s.c3;
    mx = mx > s.k1 + 1 ? mx : s.k1 + 1;
    s.cpad = (int)align_up(mx, 128);
    s.ctas = cta_budget(a);
    s.deterministic = a.deterministic != 0;
    return s;
}

constexpr int MAX_GX = 160;  // >= SM count: CTAs writing per-CTA partial buffers (4 slots each)

// 1 when b2pn_sa_forward runs these arguments through the single-launch evaluation kernel if h1 == NULL (no hidden
// activations stored)
int sa_eval_fused_bf16(const b2pn_sa_args &a)
{
    if (a.mlp.c[0] != a.c_in + 3) return 0;
    const ShapesTC s = shapes_tc(a);
    return !a.training && chain_shapes_ok(a, s.k1, s.c1, s.c2, s.c3) ? 1 : 0;
}

static int check_args_tc(const b2pn_sa_args &a)
{
    if (a.n_src < 0 || a.n_dst < 0 || a.c_in < 0) return B2PN_EINVAL;
    if (a.mlp.c[0] != a.c_in + 3 || a.mlp.c[1] <= 0 || a.mlp.c[2] <= 0 || a.mlp.c[3] <= 0) return B2PN_EINVAL;
    if (a.mlp.act != B2PN_ACT_NONE && a.mlp.act != B2PN_ACT_RELU) return B2PN_ENOTSUP;
    if (a.x_dtype != B2PN_X_F32 && a.x_dtype != B2PN_X_BF16) return B2PN_EINVAL;
    if (a.seg_mode == B2PN_SEG_SLOTS) {
        if (a.K <= 0) return B2PN_EINVAL;
        if (a.K > 64) return B2PN_ENOTSUP;  // a centroid's rows must fit one 64-column epilogue scan
        if (a.n_dst > 0 && (!a.nbr || !a.cnt || !a.pos_dst)) return B2PN_EINVAL;
        // compacted rows from b2pn_pack_rows
        if (a.n_dst > 0 && (!a.rgrp || !a.row_src || !a.num_rows)) return B2PN_EINVAL;
        if (a.n_dst > 0 && a.row_capacity < b2pn_pack_rows_capacity(a.n_dst, a.K)) return B2PN_EINVAL;
    } else if (a.seg_mode == B2PN_SEG_CLOUDS) {
        if (a.n_src > 0 && !a.batch) return B2PN_EINVAL;
    } else {
        return B2PN_EINVAL;
    }
    if (a.n_src > 0 && (!a.pos_src || (a.c_in > 0 && !a.x))) return B2PN_EINVAL;
    for (int l = 0; l < 3; ++l)
        if (!a.mlp.w[l] || !a.mlp.b[l]) return B2PN_EINVAL;
    for (int l = 0; l < 2; ++l)
        if (!a.mlp.gamma[l] || !a.mlp.beta[l] || !a.mlp.running_mean[l] || !a.mlp.running_var[l]) return B2PN_EINVAL;
    if (!a.out) return B2PN_EINVAL;
    // the arg-max slots and the hidden-activation buffers are only touched by the multi-pass (training / wide-level) kernels
    if (!(a.h1 == nullptr && sa_eval_fused_bf16(a)) && (!a.arg || !a.h1 || !a.h2 || !a.bn || !a.a1 || !a.a2)) return B2PN_EINVAL;
    return B2PN_OK;
}

static RowMapTC rowmap_tc(const b2pn_sa_args &a, const ShapesTC &s)
{
    RowMapTC rm;
    rm.seg_mode = a.seg_mode;
    rm.rgrp = a.rgrp;
    rm.row_src = a.row_src;
    rm.cnt = a.cnt;
    rm.batch = a.batch;
    rm.rows = s.rows;
    rm.n_dst = a.n_dst;
    return rm;
}
static RowsArg rowsarg_tc(const b2pn_sa_args &a, const ShapesTC &s)
{
    return RowsArg{s.rows, a.seg_mode == B2PN_SEG_SLOTS ? a.num_rows : nullptr, s.ctas};
}

struct FwdWsTC {
    Packed pk[3];
    double *partial;
    unsigned long long *keys;
};
static FwdWsTC carve_fwd_tc(const b2pn_sa_args &a, const ShapesTC &s, WsTC &ws)
{
    FwdWsTC f;
    f.pk[0] = plan_pack(s.c1, s.k1, FMT_F16);   // forward: fp16 weights meet fp16 activations
    f.pk[1] = plan_pack(s.c2, s.c1, FMT_F16);
    f.pk[2] = plan_pack(s.c3, s.c2, FMT_F16);
    for (int l = 0; l < 3; ++l) f.pk[l].img = ws.take<uint8_t>(f.pk[l].bytes);
    f.partial = ws.take<double>((int64_t)MAX_GX * 4 * 2 * s.cpad);
    f.keys = a.seg_mode == B2PN_SEG_CLOUDS ? ws.take<unsigned long long>(a.n_dst * (int64_t)s.c3) : nullptr;
    return f;
}

struct DwPlanHost {
    int MTA, num_mg, num_ng, splits, nbl_total, k_stride;
    int64_t floats;
};
// one launch covers all (row split, M group, N group) blocks; the row range is split so that the launch fills
// the GPU about once -- the partials the reduction has to read shrink with the size of dW
static DwPlanHost plan_dw(int n_out, int k_total, const ShapesTC &s)
{
    DwPlanHost d;
    const int mpad = (int)align_up(n_out, 128);
    d.MTA = mpad >= 256 ? 2 : 1;
    d.num_mg = (mpad + d.MTA * 128 - 1) / (d.MTA * 128);
    d.nbl_total = (int)align_up(k_total, 16);
    d.num_ng = (d.nbl_total + 255) / 256;
    const int64_t chunks = s.ld / 64;
    int sp = s.ctas / (d.num_mg * d.num_ng);
    if (sp < 1) sp = 1;
    if (sp > DWR_MAX_SPLITS) sp = DWR_MAX_SPLITS;
    if ((int64_t)sp > chunks) sp = (int)(chunks > 0 ? chunks : 1);
    d.splits = sp;
    d.k_stride = (int)align_up(k_total, 4);  // row stride of the partials: 16-byte aligned rows (<= nbl_total)
    d.floats = (int64_t)sp * n_out * d.k_stride;
    return d;
}

struct BwdWsTC {
    Packed pkT[3];
    double *partial;
    __nv_bfloat16 *dz1, *dz2;
    __nv_bfloat16 *dh3;  // materialised routed gradient [c3][ld]
    float *sbar;
    float *dwp[3];  // split partials of dW1, dW2, dW3 (reduced together at the end)
    long long *dxi; // deterministic mode, SLOTS levels with features: fixed-point accumulator of grad_x
};
static BwdWsTC carve_bwd_tc(const b2pn_sa_args &a, const ShapesTC &s, WsTC &ws)
{
    BwdWsTC b;
    b.pkT[2] = plan_pack(s.c2, s.c3, FMT_BF16);               // W3^T: meets gradients (bf16)
    b.pkT[1] = plan_pack(s.c1, s.c2, FMT_BF16);               // W2^T
    b.pkT[0] = plan_pack(a.c_in > 0 ? a.c_in : 1, s.c1, FMT_BF16);  // feature rows of W1^T
    for (int l = 0; l < 3; ++l) b.pkT[l].img = ws.take<uint8_t>(b.pkT[l].bytes);
    b.partial = ws.take<double>((int64_t)MAX_GX * 4 * 2 * s.cpad);
    b.dz1 = ws.take<__nv_bfloat16>((int64_t)s.c1 * s.ld);
    b.dz2 = ws.take<__nv_bfloat16>((int64_t)s.c2 * s.ld);
    // the dense routed gradient exists only at the global level (SLOTS levels generate it on the fly)
    b.dh3 = a.seg_mode == B2PN_SEG_CLOUDS ? ws.take<__nv_bfloat16>((int64_t)s.c3 * s.ld) : nullptr;
    b.sbar = ws.take<float>(2 * s.cmax);
    b.dwp[2] = ws.take<float>(plan_dw(s.c3, s.c2 + 1, s).floats);
    b.dwp[1] = ws.take<float>(plan_dw(s.c2, s.c1 + 1, s).floats);
    b.dwp[0] = ws.take<float>(plan_dw(s.c1, s.k1 + 1, s).floats);
    b.dxi = (s.deterministic && a.seg_mode == B2PN_SEG_SLOTS && a.c_in > 0) ? ws.take<long long>(a.n_src * (int64_t)a.c_in) : nullptr;
    return b;
}

int64_t sa_workspace_bytes_bf16(const b2pn_sa_args &a, int backward)
{
    const ShapesTC s = shapes_tc(a);
    WsTC ws(nullptr);
    if (backward) carve_bwd_tc(a, s, ws);
    else carve_fwd_tc(a, s, ws);
    return ws.off + 2048;
}

// layer-1 operand through the materialised tensor g1 (SLOTS levels whose image fits one dW N group)
static bool l1_materialised(const b2pn_sa_args &a, const ShapesTC &s)
{
    return a.seg_mode == B2PN_SEG_SLOTS && a.g1 != nullptr && s.k1 + 1 + 15 <= 256;
}

static void launch_gather_l1(const b2pn_sa_args &a, const ShapesTC &s, cudaStream_t st)
{
    const RowMapTC rm = rowmap_tc(a, s);
    const RowsArg ra = rowsarg_tc(a, s);
    GatherLoaderTC gg = {rm, a.x, s.cols, a.pos_src, a.pos_dst, s.k1, FMT_F16};  // column k1 = ones (dW1 bias line)
    const int kg = s.k1 + 1, kg8 = (kg + 7) & ~7;
    gather_l1_tc_kernel<<<(unsigned)(s.ld / GATHER_ROWS), 256, kg8 * GATHER_ROWS * 2, st>>>(gg, ra.dev, kg, s.ld,
                                                                                             (__nv_bfloat16 *)a.g1);
    note_launch();
}

// b2pn_sa_gather_rows: the gather alone (geometry + raw inputs only; include/b2pn.h)
int sa_gather_rows_bf16(const b2pn_sa_args &a, cudaStream_t st)
{
    if (a.n_src < 0 || a.n_dst < 0 || a.c_in < 0 || a.mlp.c[0] != a.c_in + 3) return B2PN_EINVAL;
    if (a.x_dtype != B2PN_X_F32 && a.x_dtype != B2PN_X_BF16) return B2PN_EINVAL;
    if (a.seg_mode != B2PN_SEG_SLOTS) return B2PN_ENOTSUP;
    if (a.K <= 0) return B2PN_EINVAL;
    if (a.K > 64) return B2PN_ENOTSUP;
    if (a.n_dst == 0) return B2PN_OK;
    if (!a.pos_dst || !a.pos_src || (a.c_in > 0 && !a.x) || !a.rgrp || !a.row_src || !a.num_rows) return B2PN_EINVAL;
    if (a.row_capacity < b2pn_pack_rows_capacity(a.n_dst, a.K)) return B2PN_EINVAL;
    const ShapesTC s = shapes_tc(a);
    if (!l1_materialised(a, s)) return a.g1 ? B2PN_ENOTSUP : B2PN_EINVAL;
    launch_gather_l1(a, s, st);
    B2PN_LAUNCH_CHECK();
    return B2PN_OK;
}

// BatchNorm layer l (0 or 1) of the forward: batch statistics from `nparts` partial slices (training) or the running
// statistics -> its rows [mean, rstd, scale, shift] of the bn buffer
static void launch_bn_fwd_finalize(const b2pn_sa_args &a, const ShapesTC &s, int l, const double *partial, int nparts,
                                   const CountArg &count, cudaStream_t st)
{
    const int C = l == 0 ? s.c1 : s.c2;
    bn_fwd_finalize_tc_kernel<<<(C + 3) / 4, 128, 0, st>>>(partial, nparts, C, s.cpad, count, a.training, a.mlp.b[l], a.mlp.gamma[l],
                                                           a.mlp.beta[l], a.mlp.running_mean[l], a.mlp.running_var[l],
                                                           a.mlp.num_batches_tracked[l], a.mlp.eps, a.mlp.momentum,
                                                           a.bn + l * 4 * s.cmax, s.cmax);
    note_launch();
}

// grid of a chained kernel (sa_chain.cuh) over `tiles64` tiles of 64 rows: CH_SLOTS tiles per CTA and round, at most the
// call's CTA budget
static int chain_grid(const ShapesTC &s, int64_t tiles64)
{
    const int64_t need = (tiles64 + CH_SLOTS - 1) / CH_SLOTS;
    return need < s.ctas ? (int)need : s.ctas;
}

// one launch of a chained kernel; its dynamic shared memory is raised once per device (ensure_dynamic_smem)
template <auto KERN, class... Args>
static int launch_chain(int gx, int threads, int smem, cudaStream_t st, const Args &...args)
{
    static SmemAttrSlot slot = {};
    cudaError_t e = ensure_dynamic_smem(KERN, smem, slot);
    if (e != cudaSuccess) return (int)e;
    KERN<<<gx, threads, smem, st>>>(args...);
    note_launch();
    e = cudaPeekAtLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

int sa_forward_bf16(const b2pn_sa_args &a, cudaStream_t st)
{
    int rc = check_args_tc(a);
    if (rc) return rc;
    const ShapesTC s = shapes_tc(a);
    if (a.n_dst == 0) return B2PN_OK;
    if (a.workspace_bytes < sa_workspace_bytes_bf16(a, 0) || !a.workspace) return B2PN_EINVAL;
    WsTC ws(a.workspace);
    FwdWsTC f = carve_fwd_tc(a, s, ws);
    const RowMapTC rm = rowmap_tc(a, s);
    const RowsArg ra = rowsarg_tc(a, s);
    __nv_bfloat16 *z1 = (__nv_bfloat16 *)a.h1, *z2 = (__nv_bfloat16 *)a.h2;
    float *bn1 = a.bn, *bn2 = a.bn + 4 * s.cmax;
    const int train = a.training;

    // (the chained training kernels read g1 with its ones line)
    const bool train_chain = a.training && s.rows > 0 && l1_materialised(a, s) && chain_shapes_ok(a, s.k1 + 1, s.c1, s.c2, s.c3);
    {
        PackJob jobs[3] = {pack_job(a.mlp.w[0], s.c1, s.k1, s.c0, 1, &s.cols, f.pk[0]),
                           pack_job(a.mlp.w[1], s.c2, s.c1, s.c1, 1, nullptr, f.pk[1]),
                           pack_job(a.mlp.w[2], s.c3, s.c2, s.c2, 1, nullptr, f.pk[2])};
        // chained training passes: a 64-channel hidden layer leaves half of the 128 accumulator lanes empty; its image
        // repeats the 64 rows so that the normalising epilogue runs on all eight warps (every other consumer of these
        // images ignores lanes past the layer's width)
        jobs[0].dup64 = train_chain && s.c1 == 64;
        jobs[1].dup64 = train_chain && s.c2 == 64;
        launch_packs(jobs, 3, st);
    }
    if (a.h1 == nullptr && sa_eval_fused_bf16(a)) {
        // evaluation mode: the whole level in one launch, nothing but `out` written (sa_chain.cuh)
        if (s.rows == 0) return B2PN_OK;
        ChainParams cp = {};
        for (int l = 0; l < 3; ++l) {
            cp.w_img[l] = f.pk[l].img;
            cp.w_bytes[l] = (int)f.pk[l].bytes;
            cp.bias[l] = a.mlp.b[l];
        }
        for (int l = 0; l < 2; ++l) {
            cp.gamma[l] = a.mlp.gamma[l];
            cp.beta[l] = a.mlp.beta[l];
            cp.mean[l] = a.mlp.running_mean[l];
            cp.var[l] = a.mlp.running_var[l];
        }
        cp.k_img = s.k1;
        cp.k1c = f.pk[0].num_kc;
        cp.c1c = f.pk[1].num_kc;
        cp.c2c = f.pk[2].num_kc;
        cp.c1 = s.c1;
        cp.c2 = s.c2;
        cp.c3 = s.c3;
        cp.mt3 = f.pk[2].MT;
        cp.rows = ra.cap;
        cp.rows_dev = ra.dev;
        cp.eps = a.mlp.eps;
        cp.act = a.mlp.act;
        cp.out = a.out;
        cp.arg = nullptr;   // the evaluation path never differentiates through the max: the arg-max slots are not written
        cp.out16 = (__half *)a.out_bf16;
        cp.rgrp = a.rgrp;
        GatherLoaderTC cg = {rm, a.x, s.cols, a.pos_src, a.pos_dst, -1, FMT_F16};
        const int smem = chain_smem_bytes(cp);
        const int gx = chain_grid(s, (ra.cap + CH_ROWS - 1) / CH_ROWS);
        const int nks_last = (s.k1 - (cp.k1c - 1) * KC) >= KC ? 4 : (s.k1 - (cp.k1c - 1) * KC + 15) / 16;
        // the reference's two levels get fully unrolled MMA issue code; anything else the run-time-shaped instance
        if (cp.k1c == 1 && nks_last == 1 && cp.c1c == 1 && cp.c2c == 1 && cp.mt3 == 1)
            return launch_chain<tc_chain_eval_kernel<1, 1, 1, 1, 1>>(gx, CH_THREADS, smem, st, cp, cg);
        if (cp.k1c == 3 && nks_last == 1 && cp.c1c == 2 && cp.c2c == 2 && cp.mt3 == 2)
            return launch_chain<tc_chain_eval_kernel<3, 1, 2, 2, 2>>(gx, CH_THREADS, smem, st, cp, cg);
        return launch_chain<tc_chain_eval_kernel<-1, -1, -1, -1, -1>>(gx, CH_THREADS, smem, st, cp, cg);
    }
    const CountArg count = {a.seg_mode == B2PN_SEG_SLOTS ? a.num_rows + 1 : nullptr, (double)s.rows};

    // ---- layer 1: gather + concat + Linear; pass A = batch statistics, pass B = normalise + store z1
    GatherLoaderTC gl = {rm, a.x, s.cols, a.pos_src, a.pos_dst, -1, FMT_F16};
    const bool use_g1 = l1_materialised(a, s);
    TmaMap map_g1 = kNoMap;
    TmaFeatLoader tl1;
    if (use_g1 && s.rows > 0) {
        if (!a.g1_ready) launch_gather_l1(a, s, st);
        if ((rc = make_tma_feature_major(&map_g1, a.g1, s.k1 + 1, s.ld))) return rc;
    }
    const int ns1 = use_g1 ? 4 : 2;  // partial slots per CTA: 2 column halves x epilogue groups (2 when TMA-fed)
    if (train && s.rows > 0) {
        StatsEpTC<1> e1 = {s.c1, f.partial, s.cpad, ns1};
        StatsEpTC<2> e2 = {s.c1, f.partial, s.cpad, ns1};
        rc = use_g1 ? launch_by_mt(f.pk[0], ra, tl1, e1, e2, st, map_g1) : launch_by_mt(f.pk[0], ra, gl, e1, e2, st);
        if (rc) return rc;
    }
    launch_bn_fwd_finalize(a, s, 0, f.partial, ns1 * grid_x_for(f.pk[0], s.tiles, s.ctas), count, st);
    if (train_chain) {
        // ---- layers 1-3 in TWO chained launches (sa_chain.cuh): P2 normalises layer 1 and takes the statistics of layer 2
        // from the tile while it is in shared memory, P3 re-runs layer 2 on the stored a1, normalises, and runs layer 3 + max
        const int gx = chain_grid(s, s.tiles * 2);   // whole 128-row tiles
        // output maps of zhat / a: boxes of 64 rows x 64 channels, the layout of the shared-memory tiles
        TmaMap mz1, ma1, mz2, ma2;
        if ((rc = make_tma_feature_major(&mz1, z1, s.c1, s.ld)) || (rc = make_tma_feature_major(&ma1, a.a1, s.c1, s.ld)) ||
            (rc = make_tma_feature_major(&mz2, z2, s.c2, s.ld)) || (rc = make_tma_feature_major(&ma2, a.a2, s.c2, s.ld)))
            return rc;
        ChainTrainParams p2 = {};
        p2.w_img[0] = f.pk[0].img; p2.w_bytes[0] = (int)f.pk[0].bytes;
        p2.w_img[1] = f.pk[1].img; p2.w_bytes[1] = (int)f.pk[1].bytes;
        p2.k_in = s.k1; p2.kc_in = f.pk[0].num_kc; p2.kc_mid = f.pk[1].num_kc;
        p2.c_a = s.c1; p2.c_b = s.c2; p2.mt_b = 1; p2.dup_a = s.c1 == 64;
        p2.rows = ra.cap; p2.rows_dev = ra.dev; p2.ld = s.ld;
        p2.bias_a = a.mlp.b[0]; p2.mean_a = bn1; p2.rstd_a = bn1 + s.cmax; p2.gamma_a = a.mlp.gamma[0]; p2.beta_a = a.mlp.beta[0];
        p2.act = a.mlp.act; p2.z_out = (__half *)z1; p2.a_out = (__half *)a.a1;
        p2.partial = f.partial; p2.cpad = s.cpad; p2.rgrp = a.rgrp;
        const int smem2 = chain_train_smem_bytes(p2);
        const int nks1 = (s.k1 - (p2.kc_in - 1) * KC) >= KC ? 4 : (s.k1 - (p2.kc_in - 1) * KC + 15) / 16;
        if (p2.kc_in == 1 && nks1 == 1 && p2.kc_mid == 1)
            rc = launch_chain<tc_chain_train_kernel<2, 1, 1, 1, 1>>(gx, CT_THREADS, smem2, st, p2, map_g1, mz1, ma1);
        else if (p2.kc_in == 3 && nks1 == 1 && p2.kc_mid == 2)
            rc = launch_chain<tc_chain_train_kernel<2, 3, 1, 2, 1>>(gx, CT_THREADS, smem2, st, p2, map_g1, mz1, ma1);
        else
            rc = launch_chain<tc_chain_train_kernel<2, -1, -1, -1, -1>>(gx, CT_THREADS, smem2, st, p2, map_g1, mz1, ma1);
        if (rc) return rc;
        launch_bn_fwd_finalize(a, s, 1, f.partial, 4 * gx, count, st);
        TmaMap map_in3;   // P3 reads a1
        if ((rc = make_tma_feature_major(&map_in3, a.a1, s.c1, s.ld))) return rc;
        ChainTrainParams p3 = {};
        p3.w_img[0] = f.pk[1].img; p3.w_bytes[0] = (int)f.pk[1].bytes;
        p3.w_img[1] = f.pk[2].img; p3.w_bytes[1] = (int)f.pk[2].bytes;
        p3.k_in = s.c1; p3.kc_in = f.pk[1].num_kc; p3.kc_mid = f.pk[2].num_kc;
        p3.c_a = s.c2; p3.c_b = s.c3; p3.mt_b = f.pk[2].MT; p3.dup_a = s.c2 == 64;
        p3.rows = ra.cap; p3.rows_dev = ra.dev; p3.ld = s.ld;
        p3.bias_a = a.mlp.b[1]; p3.mean_a = bn2; p3.rstd_a = bn2 + s.cmax; p3.gamma_a = a.mlp.gamma[1]; p3.beta_a = a.mlp.beta[1];
        p3.act = a.mlp.act; p3.z_out = (__half *)z2; p3.a_out = (__half *)a.a2;
        p3.bias_b = a.mlp.b[2]; p3.out = a.out; p3.arg = a.arg; p3.out16 = (__half *)a.out_bf16; p3.rgrp = a.rgrp;
        const int smem3 = chain_train_smem_bytes(p3);
        if (p3.kc_in == 1 && p3.kc_mid == 1 && p3.mt_b == 1)
            return launch_chain<tc_chain_train_kernel<3, 1, 4, 1, 1>>(gx, CT_THREADS, smem3, st, p3, map_in3, mz2, ma2);
        if (p3.kc_in == 2 && p3.kc_mid == 2 && p3.mt_b == 2)
            return launch_chain<tc_chain_train_kernel<3, 2, 4, 2, 2>>(gx, CT_THREADS, smem3, st, p3, map_in3, mz2, ma2);
        return launch_chain<tc_chain_train_kernel<3, -1, -1, -1, -1>>(gx, CT_THREADS, smem3, st, p3, map_in3, mz2, ma2);
    }
    if (s.rows > 0) {
        NormStoreEpTC e = {s.c1, a.mlp.b[0], bn1, bn1 + s.cmax, a.mlp.gamma[0], a.mlp.beta[0], a.mlp.act, rm};
        TmaMap mz, ma;  // 32-channel boxes: one per epilogue warp
        if ((rc = make_tma_feature_major(&mz, z1, s.c1, s.ld, 32))) return rc;
        if ((rc = make_tma_feature_major(&ma, a.a1, s.c1, s.ld, 32))) return rc;
        rc = use_g1 ? launch_by_mt(f.pk[0], ra, tl1, e, e, st, map_g1, mz, ma) : launch_by_mt(f.pk[0], ra, gl, e, e, st, kNoMap, mz, ma);
        if (rc) return rc;
    }
    // ---- layer 2
    // layers 2 and 3 read the stored activations a1 / a2 through the TMA unit (no loader arithmetic)
    TmaFeatLoader l2, l3;
    TmaMap map_a1, map_a2;
    if ((rc = make_tma_feature_major(&map_a1, a.a1, s.c1, s.ld))) return rc;
    if ((rc = make_tma_feature_major(&map_a2, a.a2, s.c2, s.ld))) return rc;
    if (train && s.rows > 0) {
        StatsEpTC<1> e1 = {s.c2, f.partial, s.cpad, 4};
        StatsEpTC<2> e2 = {s.c2, f.partial, s.cpad, 4};
        if ((rc = launch_by_mt(f.pk[1], ra, l2, e1, e2, st, map_a1))) return rc;
    }
    launch_bn_fwd_finalize(a, s, 1, f.partial, 4 * grid_x_for(f.pk[1], s.tiles, s.ctas), count, st);
    if (s.rows > 0) {
        NormStoreEpTC e = {s.c2, a.mlp.b[1], bn2, bn2 + s.cmax, a.mlp.gamma[1], a.mlp.beta[1], a.mlp.act, rm};
        TmaMap mz, ma;
        if ((rc = make_tma_feature_major(&mz, z2, s.c2, s.ld, 32))) return rc;
        if ((rc = make_tma_feature_major(&ma, a.a2, s.c2, s.ld, 32))) return rc;
        if ((rc = launch_by_mt(f.pk[1], ra, l2, e, e, st, map_a1, mz, ma))) return rc;
    }
    // ---- layer 3 + max aggregation
    if (a.seg_mode == B2PN_SEG_SLOTS) {
        SlotMaxEpTC e = {a.out, a.arg, s.c3, a.mlp.b[2], a.rgrp, s.rows, (__half *)a.out_bf16};
        if ((rc = launch_by_mt(f.pk[2], ra, l3, e, e, st, map_a2))) return rc;
    } else {
        const int64_t n = a.n_dst * (int64_t)s.c3;
        B2PN_CUDA(cudaMemsetAsync(f.keys, 0, n * sizeof(unsigned long long), st));
        if (s.rows > 0) {
            CloudMaxEpTC e = {f.keys, s.c3, a.mlp.b[2], a.batch, s.rows};
            if ((rc = launch_by_mt(f.pk[2], ra, l3, e, e, st, map_a2))) return rc;
        }
        unpack_keys_tc_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(f.keys, a.out, a.arg, n);
        note_launch();
    }
    B2PN_LAUNCH_CHECK();
    return B2PN_OK;
}

template <class YS, class XF>
static int launch_dw(const YS &ys, const XF &xf, int n_out, int k_total, const ShapesTC &s, const RowsArg &ra, float *dwp,
                     cudaStream_t st, const TmaMap &map_y = kNoMap, const TmaMap &map_x = kNoMap, const TmaMap &map_v = kNoMap)
{
    const DwPlanHost d = plan_dw(n_out, k_total, s);
    DwParams p = {ra.cap, ra.dev, n_out, d.nbl_total, d.k_stride, dwp, s.deterministic ? 0 : 1, 0, 0};
    if (!s.deterministic) {
        cudaError_t em = cudaMemsetAsync(dwp, 0, (size_t)n_out * d.k_stride * sizeof(float), st);
        if (em != cudaSuccess) return (int)em;
    }
    const int nb_max = d.nbl_total < 256 ? d.nbl_total : 256;
    const int b_bytes = (int)align_up(XF::bytes(nb_max), 1024);
    dim3 grid((unsigned)d.splits, (unsigned)d.num_mg, (unsigned)d.num_ng);
    cudaError_t e;
    auto plan = [&](int a_bytes) {
        p.stage_bytes = a_bytes + b_bytes;
        p.stages = (DwPlan<1>::SMEM_BUDGET - 1280) / p.stage_bytes;
        if (p.stages > DwPlan<1>::MAX_STAGES) p.stages = DwPlan<1>::MAX_STAGES;
        if (p.stages < 2) p.stages = 2;
        return p.stages * p.stage_bytes + 256 + 1024;
    };
    if (d.MTA == 1) {
        auto kern = tc_dw_kernel<1, YS, XF>;
        const int smem = plan(DwPlan<1>::A_BYTES);
        static SmemAttrSlot slot = {};
        e = ensure_dynamic_smem(kern, smem, slot);
        if (e != cudaSuccess) return (int)e;
        kern<<<grid, NT, smem, st>>>(p, ys, xf, map_y, map_x, map_v);
    } else {
        auto kern = tc_dw_kernel<2, YS, XF>;
        const int smem = plan(DwPlan<2>::A_BYTES);
        static SmemAttrSlot slot = {};
        e = ensure_dynamic_smem(kern, smem, slot);
        if (e != cudaSuccess) return (int)e;
        kern<<<grid, NT, smem, st>>>(p, ys, xf, map_y, map_x, map_v);
    }
    note_launch();
    e = cudaPeekAtLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

// grid of the element-wise BN-backward pass: grid-stride, at most 8 blocks of 256 threads per SM
static unsigned apply_grid(const ShapesTC &s, int C)
{
    const int64_t n = (s.ld / 8) * C;
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)s.ctas * 8;
    if (blocks > cap) blocks = cap;
    return (unsigned)(blocks > 0 ? blocks : 1);
}

static DwReduceJob dw_reduce_job(const float *dwp, int n_out, int k_total, const InCols *map, int k_true, int ones_idx,
                                 const ShapesTC &s, float *gw, float *gb)
{
    const DwPlanHost d = plan_dw(n_out, k_total, s);
    DwReduceJob j = {dwp, s.deterministic ? d.splits : 1, n_out, d.k_stride, map ? 1 : 0, map ? *map : InCols{0, 0}, k_true, ones_idx, gw, gb};
    return j;
}
static void launch_dw_reduces(const DwReduceJob *jobs, int n, cudaStream_t st)
{
    DwReduceJobs dj;
    int64_t mx = 0;
    for (int i = 0; i < 3; ++i) {
        dj.j[i] = jobs[i < n ? i : 0];
        const int64_t tot = (int64_t)dj.j[i].n_out * (dj.j[i].k_true + 1);
        mx = tot > mx ? tot : mx;
    }
    if (mx <= 16384)
        dw_reduce_tc_kernel<<<dim3((unsigned)((mx + 31) / 32), (unsigned)n), dim3(32, DWR_WARPS), 0, st>>>(dj);
    else
        dw_reduce_flat_tc_kernel<<<dim3((unsigned)((mx + 127) / 128), (unsigned)n), 128, 0, st>>>(dj);
    note_launch();
}

int sa_backward_bf16(const b2pn_sa_args &a, const b2pn_sa_grads &g, cudaStream_t st)
{
    int rc = check_args_tc(a);
    if (rc) return rc;
    if (!g.grad_out) return B2PN_EINVAL;
    const ShapesTC s = shapes_tc(a);
    if (a.n_dst == 0 || s.rows == 0) return B2PN_OK;
    if (a.workspace_bytes < sa_workspace_bytes_bf16(a, 1) || !a.workspace) return B2PN_EINVAL;
    WsTC ws(a.workspace);
    BwdWsTC b = carve_bwd_tc(a, s, ws);
    const RowMapTC rm = rowmap_tc(a, s);
    const RowsArg ra = rowsarg_tc(a, s);
    const __nv_bfloat16 *z1 = (const __nv_bfloat16 *)a.h1, *z2 = (const __nv_bfloat16 *)a.h2;
    float *bn1 = a.bn, *bn2 = a.bn + 4 * s.cmax;
    const bool need_dx = g.grad_x != nullptr && a.c_in > 0;

    {
        const PackJob jobs[3] = {pack_job(a.mlp.w[2], s.c2, s.c3, 1, s.c2, nullptr, b.pkT[2]),  // (m, k) = W3[k][m]
                                 pack_job(a.mlp.w[1], s.c1, s.c2, 1, s.c1, nullptr, b.pkT[1]),
                                 pack_job(a.mlp.w[0], a.c_in, s.c1, 1, s.c0, nullptr, b.pkT[0])};
        launch_packs(jobs, need_dx ? 3 : 2, st);
    }
    const CountArg count = {a.seg_mode == B2PN_SEG_SLOTS ? a.num_rows + 1 : nullptr, (double)s.rows};

    // ---- layer 3 ---------------------------------------------------------------------------------------
    MaskSumsStoreEpTC<1> e31 = {s.c2, a.mlp.gamma[1], a.mlp.beta[1], a.mlp.act, b.partial, s.cpad, 4};
    MaskSumsStoreEpTC<2> e32 = {s.c2, a.mlp.gamma[1], a.mlp.beta[1], a.mlp.act, b.partial, s.cpad, 4};
    TmaMap mdz2, mz2;  // epilogue maps (32-channel boxes): dz2 out, zhat2 in
    if ((rc = make_tma_feature_major(&mdz2, b.dz2, s.c2, s.ld, 32))) return rc;
    if ((rc = make_tma_feature_major(&mz2, z2, s.c2, s.ld, 32))) return rc;
    LineFillK<FeatSource<1>> xa2 = {{rm, z2, s.c2, s.ld, a.mlp.act, s.c2, a.mlp.gamma[1], a.mlp.beta[1], FMT_BF16}};
    // X sides through TMA: stored activations + the row-valid "ones" line (64-channel boxes, so c % 64 == 0)
    TmaMap map_v = kNoMap, map_a1 = kNoMap, map_a2 = kNoMap;
    const bool tma_x = a.row_valid != nullptr;
    const bool tma_x2 = tma_x && s.c2 % 64 == 0 && (s.c2 % 256) + 16 <= 256, tma_x1 = tma_x && s.c1 % 64 == 0 && (s.c1 % 256) + 16 <= 256;
    if (tma_x2 || tma_x1) {
        if ((rc = make_tma_row_valid(&map_v, a.row_valid, s.ld))) return rc;
    }
    if (tma_x2 && (rc = make_tma_feature_major(&map_a2, a.a2, s.c2, s.ld))) return rc;
    if (tma_x1 && (rc = make_tma_feature_major(&map_a1, a.a1, s.c1, s.ld))) return rc;
    if (a.seg_mode == B2PN_SEG_CLOUDS) {
        // global level (few rows): materialise dh3 once, then both consumers read it through TMA
        route_grad_clouds_tc_kernel<<<apply_grid(s, s.c3), 256, 0, st>>>(rm, ra.dev, g.grad_out, a.arg, s.c3, s.ld, b.dh3);
        note_launch();
        TmaMap map3;
        if ((rc = make_tma_feature_major(&map3, b.dh3, s.c3, s.ld))) return rc;
        TmaFeatLoader bl;
        if ((rc = launch_by_mt(b.pkT[2], ra, bl, e31, e32, st, map3, mdz2, mz2))) return rc;          // da2 = W3^T dh3
        TmaSource y3 = {rm};
        if (tma_x2) {
            TmaFill xt = {s.c2, 1};
            rc = launch_dw(y3, xt, s.c3, s.c2 + 1, s, ra, b.dwp[2], st, map3, map_a2, map_v);   // dW3 = dh3^T a2
        } else {
            rc = launch_dw(y3, xa2, s.c3, s.c2 + 1, s, ra, b.dwp[2], st, map3);
        }
        if (rc) return rc;
    } else {
        // SLOTS levels: dh3 is one value per (centroid, channel) -- both consumers generate their operand tiles from
        // (arg, grad_out) in their loader warps instead of streaming a dense [c3][rows] tensor
        const int vec = (s.c3 % 4 == 0 && ((uintptr_t)g.grad_out | (uintptr_t)a.arg) % 16 == 0) ? 1 : 0;
        RouteSource rs = {rm, g.grad_out, a.arg, s.c3, vec};
        FeatLoaderTC<RouteSource, true> bl = {rs};
        if ((rc = launch_by_mt(b.pkT[2], ra, bl, e31, e32, st, kNoMap, mdz2, mz2))) return rc;        // da2 = W3^T dh3
        if (tma_x2) {
            TmaFill xt = {s.c2, 1};
            rc = launch_dw(rs, xt, s.c3, s.c2 + 1, s, ra, b.dwp[2], st, kNoMap, map_a2, map_v);  // dW3 = dh3^T a2
        } else {
            rc = launch_dw(rs, xa2, s.c3, s.c2 + 1, s, ra, b.dwp[2], st);
        }
        if (rc) return rc;
    }
    bn_bwd_finalize_tc_kernel<<<(s.c2 + 3) / 4, 128, 0, st>>>(b.partial, 4 * grid_x_for(b.pkT[2], s.tiles, s.ctas), s.c2, s.cpad, count,
                                                                 a.training, g.grad_gamma[1], g.grad_beta[1], b.sbar);
    note_launch();
    {
        bn_bwd_apply_tc_kernel<<<apply_grid(s, s.c2), 256, 0, st>>>(rm, ra.dev, b.dz2, z2, s.c2, s.ld, bn2 + 2 * s.cmax, b.sbar);
        note_launch();
    }
    // ---- layer 2 ---------------------------------------------------------------------------------------
    // dh2 / dh1 are plain stored tensors by now (invalid rows zeroed by the BN-backward pass): the TMA unit feeds them
    TmaMap map2, map1;
    if ((rc = make_tma_feature_major(&map2, b.dz2, s.c2, s.ld))) return rc;
    if ((rc = make_tma_feature_major(&map1, b.dz1, s.c1, s.ld))) return rc;
    TmaSource y2 = {rm};
    {
        TmaFeatLoader bl;
        MaskSumsStoreEpTC<1> e1 = {s.c1, a.mlp.gamma[0], a.mlp.beta[0], a.mlp.act, b.partial, s.cpad, 4};
        MaskSumsStoreEpTC<2> e2 = {s.c1, a.mlp.gamma[0], a.mlp.beta[0], a.mlp.act, b.partial, s.cpad, 4};
        TmaMap mdz1, mz1;
        if ((rc = make_tma_feature_major(&mdz1, b.dz1, s.c1, s.ld, 32))) return rc;
        if ((rc = make_tma_feature_major(&mz1, z1, s.c1, s.ld, 32))) return rc;
        if ((rc = launch_by_mt(b.pkT[1], ra, bl, e1, e2, st, map2, mdz1, mz1))) return rc;
        if (tma_x1) {
            TmaFill xt = {s.c1, 1};
            rc = launch_dw(y2, xt, s.c2, s.c1 + 1, s, ra, b.dwp[1], st, map2, map_a1, map_v);
        } else {
            LineFillK<FeatSource<1>> xa1 = {{rm, z1, s.c1, s.ld, a.mlp.act, s.c1, a.mlp.gamma[0], a.mlp.beta[0], FMT_BF16}};
            rc = launch_dw(y2, xa1, s.c2, s.c1 + 1, s, ra, b.dwp[1], st, map2);
        }
        if (rc) return rc;
    }
    bn_bwd_finalize_tc_kernel<<<(s.c1 + 3) / 4, 128, 0, st>>>(b.partial, 4 * grid_x_for(b.pkT[1], s.tiles, s.ctas), s.c1, s.cpad, count,
                                                                 a.training, g.grad_gamma[0], g.grad_beta[0], b.sbar);
    note_launch();
    {
        bn_bwd_apply_tc_kernel<<<apply_grid(s, s.c1), 256, 0, st>>>(rm, ra.dev, b.dz1, z1, s.c1, s.ld, bn1 + 2 * s.cmax, b.sbar);
        note_launch();
    }
    // ---- layer 1 ---------------------------------------------------------------------------------------
    TmaSource y1 = {rm};
    {
        if (l1_materialised(a, s)) {
            TmaMap map_g1;
            if ((rc = make_tma_feature_major(&map_g1, a.g1, s.k1 + 1, s.ld))) return rc;
            TmaFill xt = {s.k1 + 1, 0};
            rc = launch_dw(y1, xt, s.c1, s.k1 + 1, s, ra, b.dwp[0], st, map1, map_g1, kNoMap);
        } else {
            LineFillGather xg = {{rm, a.x, s.cols, a.pos_src, a.pos_dst, s.k1, FMT_BF16}};  // X side of dW1: meets bf16 gradients
            rc = launch_dw(y1, xg, s.c1, s.k1 + 1, s, ra, b.dwp[0], st, map1);
        }
        if (rc) return rc;
        const DwReduceJob jobs[3] = {dw_reduce_job(b.dwp[2], s.c3, s.c2 + 1, nullptr, s.c2, s.c2, s, g.grad_w[2], g.grad_b[2]),
                                     dw_reduce_job(b.dwp[1], s.c2, s.c1 + 1, nullptr, s.c1, s.c1, s, g.grad_w[1], g.grad_b[1]),
                                     dw_reduce_job(b.dwp[0], s.c1, s.k1 + 1, &s.cols, s.c0, s.k1, s, g.grad_w[0], g.grad_b[0])};
        launch_dw_reduces(jobs, 3, st);
    }
    if (need_dx) {
        TmaFeatLoader bl;
        const int64_t nx = a.n_src * (int64_t)a.c_in;
        // the scatter-add target starts from zero (SLOTS levels; CLOUDS levels store every row exactly once)
        if (b.dxi) B2PN_CUDA(cudaMemsetAsync(b.dxi, 0, (size_t)nx * sizeof(long long), st));
        else if (a.seg_mode == B2PN_SEG_SLOTS) B2PN_CUDA(cudaMemsetAsync(g.grad_x, 0, (size_t)nx * sizeof(float), st));
        ScatterEpTC e = {rm, g.grad_x, a.c_in, b.dxi};
        if ((rc = launch_by_mt(b.pkT[0], ra, bl, e, e, st, map1))) return rc;
        if (b.dxi) {
            fixed_to_f32_kernel<<<(unsigned)((nx + 255) / 256), 256, 0, st>>>(b.dxi, g.grad_x, nx);
            note_launch();
        }
    }
    B2PN_LAUNCH_CHECK();
    return B2PN_OK;
}

}  // namespace tc
}  // namespace b2pn
