// Regression head -- the MLP([1024, 128, 128, 4], act=None, dropout=p) behind global_max_pool
// (/root/reference/pointnet2_regressor.py:50,58; torch_geometric.nn.MLP semantics, SURVEY.md A.4):
//     Lin -> BatchNorm1d -> dropout -> Lin -> BatchNorm1d -> dropout -> Lin
// on B <= 32 rows (one row per tree cloud).  Through ATen this is ~60 tiny kernels per training step (GEMV, BN
// statistics, BN transform, dropout, their backward twins, reductions); the arithmetic is 1.7 MFLOP.  Here it is one
// forward kernel (one CTA, the batch lives in shared memory) and one backward kernel (a few CTAs: every CTA redoes the
// tiny upstream chain and then owns a slice of the 1024 input columns for dW0 / dx).  fp32 throughout.
#include <math.h>

#include "common.cuh"

namespace b2pn {

constexpr int HEAD_THREADS = 1024;
constexpr int HEAD_MAX_B = 32;
constexpr int HEAD_MAX_C = 256;   // hidden width
constexpr int HEAD_MAX_OUT = 8;

// counter-based dropout noise: one 32-bit draw per (call, layer, element); statistical parity with torch's Philox
// stream is all the reference needs (its own runs are not seed-reproducible across devices either)
__device__ __forceinline__ unsigned head_hash(unsigned long long key)
{
    key ^= key >> 33;
    key *= 0xff51afd7ed558ccdull;
    key ^= key >> 33;
    key *= 0xc4ceb9fe1a85ec53ull;
    key ^= key >> 33;
    return (unsigned)(key >> 16);
}
__device__ __forceinline__ bool head_keep(unsigned long long seed, unsigned long long call, int layer, int idx, float p)
{
    const unsigned r = head_hash(seed * 0x9e3779b97f4a7c15ull + call * 0x100000001b3ull + (unsigned long long)layer * 0x1000003ull +
                                 (unsigned long long)idx);
    return (float)(r >> 8) * (1.0f / 16777216.0f) >= p;
}

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// y[b][j] = sum_k in[b][k] * W[j][k] + bias[j]; one warp per output channel j, lanes split k; `in` in shared memory
template <int MAXB>
__device__ __forceinline__ void head_linear(const float *in, int ldin, int B, int K, const float *W, const float *bias, int J,
                                            float *out, int ldout)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int j = warp; j < J; j += nw) {
        float acc[MAXB];
#pragma unroll
        for (int b = 0; b < MAXB; ++b) acc[b] = 0.f;
        const float *w = W + (int64_t)j * K;
        for (int k = lane; k < K; k += 32) {
            const float wv = w[k];
#pragma unroll
            for (int b = 0; b < MAXB; ++b)
                if (b < B) acc[b] = fmaf(in[b * ldin + k], wv, acc[b]);
        }
        const float bj = bias[j];
#pragma unroll
        for (int b = 0; b < MAXB; ++b) {
            if (b < B) {
                const float s = warp_sum(acc[b]);
                if (lane == 0) out[b * ldout + j] = s + bj;
            }
        }
    }
}

// BatchNorm1d (+ dropout) over the B rows of channel j = thread; h -> a in place, saves xhat / mask / rstd
__device__ __forceinline__ void head_bn_dropout(float *h, int ld, int B, int C, const b2pn_head_args &a, int layer, unsigned long long call)
{
    for (int j = threadIdx.x; j < C; j += blockDim.x) {
        float mean, var;
        if (a.training) {
            float s = 0.f;
            for (int b = 0; b < B; ++b) s += h[b * ld + j];
            mean = s / (float)B;
            float q = 0.f;
            for (int b = 0; b < B; ++b) {
                const float d = h[b * ld + j] - mean;
                q = fmaf(d, d, q);
            }
            var = q / (float)B;  // biased, as BatchNorm normalises with
            const float unb = B > 1 ? q / (float)(B - 1) : var;
            a.running_mean[layer][j] = (1.f - a.momentum) * a.running_mean[layer][j] + a.momentum * mean;
            a.running_var[layer][j] = (1.f - a.momentum) * a.running_var[layer][j] + a.momentum * unb;
        } else {
            mean = a.running_mean[layer][j];
            var = a.running_var[layer][j];
        }
        const float rstd = rsqrtf(var + a.eps);
        if (a.rstd[layer]) a.rstd[layer][j] = rstd;
        const float ga = a.gamma[layer][j], be = a.beta[layer][j];
        const float keep_scale = 1.f / (1.f - a.p);
        for (int b = 0; b < B; ++b) {
            const float xh = (h[b * ld + j] - mean) * rstd;
            float y = fmaf(xh, ga, be);
            bool keep = true;
            if (a.training && a.p > 0.f) {
                keep = head_keep(a.seed, call, layer, b * C + j, a.p);
                y = keep ? y * keep_scale : 0.f;
            }
            if (a.xhat[layer]) a.xhat[layer][b * C + j] = xh;
            if (a.mask[layer]) a.mask[layer][b * C + j] = keep ? 1 : 0;
            h[b * ld + j] = y;
        }
    }
    if (threadIdx.x == 0 && a.training && a.num_batches_tracked[layer]) *a.num_batches_tracked[layer] += 1;
}

// First Linear (c0 = 1024 inputs: 512 KB of weights) spread over the GPU: one CTA per output channel, 128 threads
// split the input columns (coalesced loads of the weight row and of the B input rows, which stay cache resident).
// h1 lands in the xhat[0] buffer, which the second kernel overwrites with the normalised values.
template <int MAXB>
__global__ void __launch_bounds__(128) head_lin0_kernel(const b2pn_head_args a)
{
    __shared__ float s_part[4][MAXB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int j = blockIdx.x;
    const int B = a.B, K = a.c[0], J = a.c[1];
    float acc[MAXB];
#pragma unroll
    for (int b = 0; b < MAXB; ++b) acc[b] = 0.f;
    const float *w = a.w[0] + (int64_t)j * K;
    for (int k = threadIdx.x; k < K; k += 128) {
        const float wv = __ldg(w + k);
#pragma unroll
        for (int b = 0; b < MAXB; ++b)
            if (b < B) acc[b] = fmaf(__ldg(a.x + b * K + k), wv, acc[b]);
    }
#pragma unroll
    for (int b = 0; b < MAXB; ++b) {
        if (b < B) {
            const float s = warp_sum(acc[b]);
            if (lane == 0) s_part[warp][b] = s;
        }
    }
    __syncthreads();
    if (threadIdx.x < B) {
        const int b = threadIdx.x;
        a.xhat[0][b * J + j] = ((s_part[0][b] + s_part[1][b]) + (s_part[2][b] + s_part[3][b])) + a.b[0][j];
    }
}

// cooperative copy of n floats (16-byte aligned source, n % 4 == 0 handled by the tail loop) into shared memory
__device__ __forceinline__ void head_stage(float *dst, const float *src, int n)
{
    const int n4 = (((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0) ? (n >> 2) : 0;
    for (int i = threadIdx.x; i < n4; i += blockDim.x)
        reinterpret_cast<float4 *>(dst)[i] = __ldg(reinterpret_cast<const float4 *>(src) + i);
    for (int i = n4 * 4 + threadIdx.x; i < n; i += blockDim.x) dst[i] = __ldg(src + i);
}

// stage_w: the two small weight matrices are copied into shared memory up front (one memory latency for all of them)
// instead of being fetched row by row from L2 inside the dependent phases below
__global__ void __launch_bounds__(HEAD_THREADS, 1) head_forward_kernel(const b2pn_head_args a, int stage_w)
{
    extern __shared__ __align__(16) float hs[];
    const int B = a.B, c0 = a.c[0], c1 = a.c[1], c2 = a.c[2], c3 = a.c[3];
    float *s1 = hs;              // [B][c1]  h1 from head_lin0_kernel (parked in xhat[0])
    float *s2 = s1 + B * c1;     // [B][c2]
    float *sw1 = s2 + B * c2;    // [c2][c1] (stage_w)
    float *sw2 = sw1 + c2 * c1;  // [c3][c2] (stage_w)
    unsigned long long call = 0ull;
    if (a.rng_counter) call = (unsigned long long)*a.rng_counter;
    (void)c0;
    for (int i = threadIdx.x; i < B * c1; i += blockDim.x) s1[i] = a.xhat[0][i];
    if (stage_w) {
        head_stage(sw1, a.w[1], c2 * c1);
        head_stage(sw2, a.w[2], c3 * c2);
    }
    __syncthreads();
    head_bn_dropout(s1, c1, B, c1, a, 0, call);
    __syncthreads();
    head_linear<HEAD_MAX_B>(s1, c1, B, c1, stage_w ? sw1 : a.w[1], a.b[1], c2, s2, c2);
    __syncthreads();
    head_bn_dropout(s2, c2, B, c2, a, 1, call);
    __syncthreads();
    head_linear<HEAD_MAX_B>(s2, c2, B, c2, stage_w ? sw2 : a.w[2], a.b[2], c3, a.out, c3);
    // every thread has read the counter before anybody bumps it
    __syncthreads();
    if (threadIdx.x == 0 && a.rng_counter && a.training) *a.rng_counter += 1;
}

// ---- backward ------------------------------------------------------------------------------------------------------
// dh (pre-BN gradient) from da (gradient w.r.t. the BN+dropout output), channel j = thread; da -> dh in place
__device__ __forceinline__ void head_bn_dropout_bwd(float *d, int ld, int B, int C, const b2pn_head_args &a, int layer, float *ggamma,
                                                    float *gbeta, bool write)
{
    for (int j = threadIdx.x; j < C; j += blockDim.x) {
        const float ga = a.gamma[layer][j], rstd = a.rstd[layer][j];
        const float keep_scale = 1.f / (1.f - a.p);
        float sg = 0.f, sgx = 0.f;
        for (int b = 0; b < B; ++b) {
            float g = d[b * ld + j];
            if (a.training && a.p > 0.f) g = a.mask[layer][b * C + j] ? g * keep_scale : 0.f;
            d[b * ld + j] = g;  // gradient w.r.t. gamma*xhat+beta
            sg += g;
            sgx = fmaf(g, a.xhat[layer][b * C + j], sgx);
        }
        if (write) {
            ggamma[j] = sgx;
            gbeta[j] = sg;
        }
        for (int b = 0; b < B; ++b) {
            const float g = d[b * ld + j];
            float dh;
            if (a.training) {
                const float xh = a.xhat[layer][b * C + j];
                dh = ga * rstd * (g - sg / (float)B - xh * (sgx / (float)B));
            } else {
                dh = ga * rstd * g;
            }
            d[b * ld + j] = dh;
        }
    }
}

// activation of a hidden layer recomputed from xhat and the dropout mask
__device__ __forceinline__ float head_act(const b2pn_head_args &a, int layer, int b, int j, int C)
{
    float y = fmaf(a.xhat[layer][b * C + j], a.gamma[layer][j], a.beta[layer][j]);
    if (a.training && a.p > 0.f) y = a.mask[layer][b * C + j] ? y / (1.f - a.p) : 0.f;
    return y;
}

__global__ void __launch_bounds__(HEAD_THREADS, 1) head_backward_kernel(const b2pn_head_args a, const b2pn_head_grads g, int stage_w)
{
    extern __shared__ __align__(16) float hs[];
    const int B = a.B, c0 = a.c[0], c1 = a.c[1], c2 = a.c[2], c3 = a.c[3];
    const int cm = c1 > c2 ? c1 : c2;
    const int per = (c0 + gridDim.x - 1) / gridDim.x;  // my slice of the input columns (layer 1)
    const int k0 = blockIdx.x * per, k1 = min(c0, k0 + per);
    const int kw = k1 - k0 > 0 ? k1 - k0 : 0;
    float *sdo = hs;              // [B][c3]   dout
    float *sd2 = sdo + B * c3;    // [B][c2]   da2 -> dh2
    float *sd1 = sd2 + B * c2;    // [B][c1]   da1 -> dh1
    float *sa = sd1 + B * c1;     // [B][max(c1,c2)] recomputed activation of the layer below
    float *sw1 = sa + B * cm;     // [c2][c1]  W1                        (stage_w)
    float *sw0 = sw1 + c2 * c1;   // [c1][per] my column slice of W0     (stage_w)
    float *sx = sw0 + c1 * per;   // [B][per]  my column slice of x      (stage_w)
    const bool lead = blockIdx.x == 0;
    const int tid = threadIdx.x;
    if (stage_w) {  // everything the dependent phases below would fetch from L2 row by row: one latency, up front
        head_stage(sw1, a.w[1], c2 * c1);
        for (int i = tid; i < c1 * kw; i += blockDim.x) {
            const int j = i / kw, k = i - j * kw;
            sw0[j * per + k] = __ldg(a.w[0] + (int64_t)j * c0 + k0 + k);
        }
        for (int i = tid; i < B * kw; i += blockDim.x) {
            const int b = i / kw, k = i - b * kw;
            sx[b * per + k] = __ldg(a.x + (int64_t)b * c0 + k0 + k);
        }
    }
    for (int i = tid; i < B * c3; i += blockDim.x) sdo[i] = g.grad_out[i];
    for (int i = tid; i < B * c2; i += blockDim.x) sa[i] = head_act(a, 1, i / c2, i % c2, c2);
    __syncthreads();
    // ---- layer 3: dW2 = dout^T a2, db2, da2 = dout W2
    if (lead) {
        for (int i = tid; i < c3 * c2; i += blockDim.x) {
            const int o = i / c2, j = i - o * c2;
            float s = 0.f;
            for (int b = 0; b < B; ++b) s = fmaf(sdo[b * c3 + o], sa[b * c2 + j], s);
            g.grad_w[2][i] = s;
        }
        for (int o = tid; o < c3; o += blockDim.x) {
            float s = 0.f;
            for (int b = 0; b < B; ++b) s += sdo[b * c3 + o];
            g.grad_b[2][o] = s;
        }
    }
    for (int i = tid; i < B * c2; i += blockDim.x) {
        const int b = i / c2, j = i - b * c2;
        float s = 0.f;
        for (int o = 0; o < c3; ++o) s = fmaf(sdo[b * c3 + o], __ldg(a.w[2] + o * c2 + j), s);
        sd2[i] = s;
    }
    __syncthreads();
    head_bn_dropout_bwd(sd2, c2, B, c2, a, 1, g.grad_gamma[1], g.grad_beta[1], lead);
    __syncthreads();
    // ---- layer 2: dW1 = dh2^T a1, db1, da1 = dh2 W1
    for (int i = tid; i < B * c1; i += blockDim.x) sa[i] = head_act(a, 0, i / c1, i % c1, c1);
    __syncthreads();
    if (lead) {
        for (int i = tid; i < c2 * c1; i += blockDim.x) {
            const int o = i / c1, j = i - o * c1;
            float s = 0.f;
            for (int b = 0; b < B; ++b) s = fmaf(sd2[b * c2 + o], sa[b * c1 + j], s);
            g.grad_w[1][i] = s;
        }
        for (int o = tid; o < c2; o += blockDim.x) {
            float s = 0.f;
            for (int b = 0; b < B; ++b) s += sd2[b * c2 + o];
            g.grad_b[1][o] = s;
        }
    }
    for (int i = tid; i < B * c1; i += blockDim.x) {
        const int b = i / c1, j = i - b * c1;
        float s = 0.f;
        if (stage_w) {
            for (int o = 0; o < c2; ++o) s = fmaf(sd2[b * c2 + o], sw1[o * c1 + j], s);
        } else {
            for (int o = 0; o < c2; ++o) s = fmaf(sd2[b * c2 + o], __ldg(a.w[1] + o * c1 + j), s);
        }
        sd1[i] = s;
    }
    __syncthreads();
    head_bn_dropout_bwd(sd1, c1, B, c1, a, 0, g.grad_gamma[0], g.grad_beta[0], lead);
    __syncthreads();
    if (lead) {
        for (int o = tid; o < c1; o += blockDim.x) {
            float s = 0.f;
            for (int b = 0; b < B; ++b) s += sd1[b * c1 + o];
            g.grad_b[0][o] = s;
        }
    }
    // ---- layer 1 over my slice of the input columns: dW0[j][k] = sum_b dh1[b][j] x[b][k];  dx[b][k] = sum_j dh1[b][j] W0[j][k]
    if (kw <= 0) return;
    for (int i = tid; i < c1 * kw; i += blockDim.x) {
        const int j = i / kw, k = i - j * kw;
        float s = 0.f;
        if (stage_w) {
            for (int b = 0; b < B; ++b) s = fmaf(sd1[b * c1 + j], sx[b * per + k], s);
        } else {
            for (int b = 0; b < B; ++b) s = fmaf(sd1[b * c1 + j], __ldg(a.x + b * c0 + k0 + k), s);
        }
        g.grad_w[0][(int64_t)j * c0 + k0 + k] = s;
    }
    if (g.grad_x) {
        for (int i = tid; i < B * kw; i += blockDim.x) {
            const int b = i / kw, k = i - b * kw;
            float s = 0.f;
            if (stage_w) {
                for (int j = 0; j < c1; ++j) s = fmaf(sd1[b * c1 + j], sw0[j * per + k], s);
            } else {
                for (int j = 0; j < c1; ++j) s = fmaf(sd1[b * c1 + j], __ldg(a.w[0] + (int64_t)j * c0 + k0 + k), s);
            }
            g.grad_x[b * c0 + k0 + k] = s;
        }
    }
}

static int head_check(const b2pn_head_args &a, bool forward)
{
    if (a.B <= 0 || a.B > HEAD_MAX_B) return a.B <= 0 ? B2PN_EINVAL : B2PN_ENOTSUP;
    if (a.training && a.B < 2) return B2PN_EINVAL;  // batch statistics of one row: BatchNorm1d refuses to train on it
    if (a.c[0] <= 0 || a.c[1] <= 0 || a.c[2] <= 0 || a.c[3] <= 0) return B2PN_EINVAL;
    if (a.c[1] > HEAD_MAX_C || a.c[2] > HEAD_MAX_C || a.c[3] > HEAD_MAX_OUT) return B2PN_ENOTSUP;
    if (!(a.p >= 0.f && a.p < 1.f)) return B2PN_EINVAL;
    if (!a.x || (forward && !a.out)) return B2PN_EINVAL;
    for (int l = 0; l < 3; ++l)
        if (!a.w[l] || !a.b[l]) return B2PN_EINVAL;
    for (int l = 0; l < 2; ++l)
        if (!a.gamma[l] || !a.beta[l] || !a.running_mean[l] || !a.running_var[l]) return B2PN_EINVAL;
    return B2PN_OK;
}

}  // namespace b2pn

// ---- weighted per-component MSE (/root/reference/main.py:157-169): value and gradient in one launch -----------
namespace b2pn {
constexpr int LOSS_MAX_C = 32;
__global__ void __launch_bounds__(32) weighted_mse_kernel(const float *pred, const float *y, const float *w, int B, int C,
                                                          float *loss, float *grad)
{
    // lane c owns component c: mse_c = mean_b (y - pred)^2 summed in row order, then loss = sum_c mse_c * w_c in
    // component order (the order main.py:169 adds them up)
    const int c = threadIdx.x;
    float term = 0.f;
    if (c < C) {
        float acc = 0.f;
        const float wc = w[c], inv = 1.f / (float)B;
        for (int b = 0; b < B; ++b) {
            const float d = pred[b * C + c] - y[b * C + c];
            acc += d * d;
            if (grad) grad[b * C + c] = 2.f * wc * inv * d;
        }
        term = acc * inv * wc;
    }
    float tot = 0.f;
    for (int i = 0; i < C; ++i) tot += __shfl_sync(0xffffffffu, term, i);
    if (c == 0) *loss = tot;
}
}  // namespace b2pn

extern "C" int b2pn_weighted_mse(const float *pred, const float *y, const float *w, int32_t B, int32_t C, float *loss,
                                 float *grad, b2pn_stream_t stream)
{
    if (B <= 0 || C <= 0) return B2PN_EINVAL;
    if (C > b2pn::LOSS_MAX_C) return B2PN_ENOTSUP;
    if (!pred || !y || !w || !loss) return B2PN_EINVAL;
    b2pn::weighted_mse_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(pred, y, w, B, C, loss, grad);
    b2pn::note_launch();
    B2PN_LAUNCH_CHECK();
    return B2PN_OK;
}

extern "C" int b2pn_head_forward(const b2pn_head_args *args, b2pn_stream_t stream)
{
    using namespace b2pn;
    if (!args) return B2PN_EINVAL;
    int rc = head_check(*args, true);
    if (rc) return rc;
    const b2pn_head_args &a = *args;
    if (!a.xhat[0]) return B2PN_EINVAL;  // doubles as the scratch for the first layer's output
    const int base = a.B * (a.c[1] + a.c[2]);
    const int wts = a.c[2] * a.c[1] + a.c[3] * a.c[2];
    const int stage_w = (base + wts) * (int)sizeof(float) <= 200 * 1024 ? 1 : 0;
    const int smem = (base + (stage_w ? wts : 0)) * (int)sizeof(float);
    B2PN_CUDA(cudaFuncSetAttribute(head_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const unsigned g0 = (unsigned)a.c[1];
    if (a.B <= 16) head_lin0_kernel<16><<<g0, 128, 0, (cudaStream_t)stream>>>(a);
    else head_lin0_kernel<32><<<g0, 128, 0, (cudaStream_t)stream>>>(a);
    note_launch();
    head_forward_kernel<<<1, HEAD_THREADS, smem, (cudaStream_t)stream>>>(a, stage_w);
    note_launch();
    B2PN_LAUNCH_CHECK();
    return B2PN_OK;
}

extern "C" int b2pn_head_backward(const b2pn_head_args *args, const b2pn_head_grads *grads, b2pn_stream_t stream)
{
    using namespace b2pn;
    if (!args || !grads) return B2PN_EINVAL;
    int rc = head_check(*args, false);
    if (rc) return rc;
    const b2pn_head_args &a = *args;
    const b2pn_head_grads &g = *grads;
    if (!g.grad_out) return B2PN_EINVAL;
    for (int l = 0; l < 3; ++l)
        if (!g.grad_w[l] || !g.grad_b[l]) return B2PN_EINVAL;
    for (int l = 0; l < 2; ++l)
        if (!g.grad_gamma[l] || !g.grad_beta[l] || !a.xhat[l] || !a.rstd[l]) return B2PN_EINVAL;
    if (a.training && a.p > 0.f && (!a.mask[0] || !a.mask[1])) return B2PN_EINVAL;
    const int cm = a.c[1] > a.c[2] ? a.c[1] : a.c[2];
    int grid = (a.c[0] + 63) / 64;  // 64 input columns per CTA
    if (grid > 32) grid = 32;
    const int per = (a.c[0] + grid - 1) / grid;
    const int base = a.B * (a.c[3] + a.c[2] + a.c[1] + cm);
    const int wts = a.c[2] * a.c[1] + a.c[1] * per + a.B * per;
    const int stage_w = (base + wts) * (int)sizeof(float) <= 200 * 1024 ? 1 : 0;
    const int smem = (base + (stage_w ? wts : 0)) * (int)sizeof(float);
    B2PN_CUDA(cudaFuncSetAttribute(head_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    head_backward_kernel<<<grid, HEAD_THREADS, smem, (cudaStream_t)stream>>>(a, g, stage_w);
    note_launch();
    B2PN_LAUNCH_CHECK();
    return B2PN_OK;
}
