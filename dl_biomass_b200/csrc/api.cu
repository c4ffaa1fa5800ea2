// libb2pn: ABI bookkeeping entry points (see include/b2pn.h).
#include <math.h>

#include "common.cuh"

namespace b2pn {
long long g_launches = 0;
}

extern "C" int b2pn_abi_version(void) { return B2PN_ABI_VERSION; }

extern "C" int64_t b2pn_launch_count(void) { return (int64_t)__atomic_load_n(&b2pn::g_launches, __ATOMIC_RELAXED); }

extern "C" const char *b2pn_error_string(int code)
{
    if (code == B2PN_OK) return "ok";
    if (code == B2PN_EINVAL) return "b2pn: invalid argument (null pointer, negative size or bad flag)";
    if (code == B2PN_ENOTSUP) return "b2pn: shape not supported by the sm_100a kernels";
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "b2pn: unknown error";
}

extern "C" int64_t b2pn_fps_num_samples(int64_t n, float ratio)
{
    // torch_cluster: ceil(float32(n) * float32(ratio)); keep the product in fp32
    volatile float prod = (float)n * ratio;
    return (int64_t)ceilf(prod);
}

// ---- set-abstraction levels: precision dispatch ---------------------------------------------------
namespace b2pn {
namespace simt {
int64_t sa_workspace_bytes_f32(const b2pn_sa_args &a, int backward);
int sa_forward_f32(const b2pn_sa_args &a, cudaStream_t st);
int sa_backward_f32(const b2pn_sa_args &a, const b2pn_sa_grads &g, cudaStream_t st);
}  // namespace simt
namespace tc {
int64_t sa_workspace_bytes_bf16(const b2pn_sa_args &a, int backward);
int sa_forward_bf16(const b2pn_sa_args &a, cudaStream_t st);
int sa_gather_rows_bf16(const b2pn_sa_args &a, cudaStream_t st);
int sa_eval_fused_bf16(const b2pn_sa_args &a);
int sa_backward_bf16(const b2pn_sa_args &a, const b2pn_sa_grads &g, cudaStream_t st);
}  // namespace tc
}  // namespace b2pn

extern "C" int64_t b2pn_sa_workspace_bytes(const b2pn_sa_args *args, int32_t backward)
{
    if (!args) return B2PN_EINVAL;
    if (args->sm_limit < 0) return B2PN_EINVAL;
    if (args->precision == B2PN_PREC_F32) return b2pn::simt::sa_workspace_bytes_f32(*args, backward);
    if (args->precision == B2PN_PREC_BF16) return b2pn::tc::sa_workspace_bytes_bf16(*args, backward);
    return B2PN_ENOTSUP;
}

extern "C" int b2pn_sa_forward(const b2pn_sa_args *args, b2pn_stream_t stream)
{
    if (!args) return B2PN_EINVAL;
    if (args->sm_limit < 0) return B2PN_EINVAL;
    if (args->precision == B2PN_PREC_F32) return b2pn::simt::sa_forward_f32(*args, (cudaStream_t)stream);
    if (args->precision == B2PN_PREC_BF16) return b2pn::tc::sa_forward_bf16(*args, (cudaStream_t)stream);
    return B2PN_ENOTSUP;
}

extern "C" int b2pn_sa_eval_fused(const b2pn_sa_args *args)
{
    if (!args) return B2PN_EINVAL;
    if (args->precision != B2PN_PREC_BF16) return 0;
    return b2pn::tc::sa_eval_fused_bf16(*args);
}

extern "C" int b2pn_sa_gather_rows(const b2pn_sa_args *args, b2pn_stream_t stream)
{
    if (!args) return B2PN_EINVAL;
    if (args->precision == B2PN_PREC_BF16) return b2pn::tc::sa_gather_rows_bf16(*args, (cudaStream_t)stream);
    return B2PN_ENOTSUP;  // the fp32 kernels gather inside their loaders
}

extern "C" int b2pn_sa_backward(const b2pn_sa_args *args, const b2pn_sa_grads *grads, b2pn_stream_t stream)
{
    if (!args || !grads) return B2PN_EINVAL;
    if (args->sm_limit < 0) return B2PN_EINVAL;
    if (args->precision == B2PN_PREC_F32) return b2pn::simt::sa_backward_f32(*args, *grads, (cudaStream_t)stream);
    if (args->precision == B2PN_PREC_BF16) return b2pn::tc::sa_backward_bf16(*args, *grads, (cudaStream_t)stream);
    return B2PN_ENOTSUP;
}

// ---- tcgen05 pipeline self-test (debug aid) ---------------------------------------------------------
namespace b2pn {
namespace tc {
int tc_gemm_selftest(const float *w, int m_out, int k, const void *b, int mode, int64_t rows, int64_t ld, const float *zeros3,
                     float *out, int64_t ld_out, void *workspace, int64_t workspace_bytes, cudaStream_t st);
}
}  // namespace b2pn

extern "C" int b2pn_tc_gemm_selftest(const float *w, int32_t m_out, int32_t k, const void *b_bf16, int32_t mode, int64_t rows,
                                     int64_t ld, const float *zeros3, float *out, int64_t ld_out, void *workspace,
                                     int64_t workspace_bytes, b2pn_stream_t stream)
{
    return b2pn::tc::tc_gemm_selftest(w, m_out, k, b_bf16, mode, rows, ld, zeros3, out, ld_out, workspace, workspace_bytes,
                                      (cudaStream_t)stream);
}
