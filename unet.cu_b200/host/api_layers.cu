// Drop-in layer operators of include/unet_b200.h, section (1): the launchers of the reference's dev/*.cuh.
// Contractions (3x3 / 1x1 convolution, linear) run on the tcgen05 implicit-GEMM kernels: the fp32 NCHW operands
// are converted to NHWC bf16 in a library-owned, grow-only workspace (the reference API has no workspace argument
// apart from the split-K scratch it passes to conv2d_k3_backward2, which is ignored), the result is written back
// in the reference layout straight from the GEMM epilogue.  Memory-bound operators are exact fp32 kernels in the
// reference layout.  Shapes that violate the tensor path's divisibility rules (3-channel layers) use an exact
// fp32 direct convolution -- still a CUDA kernel of this library, never a CPU path.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <mutex>

#include "../../include/unet_b200.h"
#include "../csrc/attn_tc.cuh"
#include "../csrc/igemm.cuh"
#include "../csrc/launch.cuh"
#include "../csrc/layers_f32.cuh"
#include "../csrc/misc_ops.cuh"
#include "../csrc/nhwc_ops.cuh"
#include "host_common.h"

using namespace ub;
extern "C" void ub_count_launches(unsigned long long n);

namespace {

struct Workspace {
    void* p[8] = {nullptr};
    size_t cap[8] = {0};
    std::mutex mu;
    void* get(int slot, size_t bytes) {
        if (bytes > cap[slot]) {
            if (p[slot]) cudaFree(p[slot]);
            size_t want = bytes + bytes / 4;
            if (cudaMalloc(&p[slot], want) != cudaSuccess) {
                p[slot] = nullptr, cap[slot] = 0;
                return nullptr;
            }
            cap[slot] = want;
        }
        return p[slot];
    }
};
Workspace g_ws;

void fail(const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    ub_host_set_error(buf);
}
int finish(int launches) {
    ub_count_launches((unsigned long long)launches);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        fail("CUDA error: %s", cudaGetErrorString(e));
        return UB_ERR_CUDA;
    }
    return UB_OK;
}

// single-entry weight pack through a 1-element device table kept in workspace slot 7
int pack_one(const float* w, bf16* wf, bf16* wd, int Cout, int Cin, int ntaps, cudaStream_t st) {
    PackEntry e{w, wf, wd, Cout, Cin, ntaps};
    PackEntry* tab = (PackEntry*)g_ws.get(7, 4096);
    if (!tab) return UB_ERR_CUDA;
    // stream-ordered upload of 40 bytes (pageable source is copied synchronously into the driver's staging buffer)
    if (cudaMemcpyAsync(tab, &e, sizeof e, cudaMemcpyHostToDevice, st) != cudaSuccess) return UB_ERR_CUDA;
    pack_weights(tab, 1, ((Cout + 31) / 32) * ((Cin + 31) / 32), st);
    return UB_OK;
}

// ub_set_layer_precision(): -1 = not yet read from the environment
int g_precision = -1;
bool fp32_mode() {
    if (g_precision < 0) {
        const char* e = getenv("UB_LAYER_PRECISION");
        g_precision = (e && (e[0] == 'f' || e[0] == 'F')) ? UB_PRECISION_FP32 : UB_PRECISION_BF16;
    }
    return g_precision == UB_PRECISION_FP32;
}
bool shape_fprop_ok(int Cin, int Cout) { return Cin % 8 == 0 && Cout % 16 == 0; }
bool shape_wgrad_ok(int Cin, int Cout) { return Cin % 64 == 0 && Cout % 64 == 0; }
bool tensor_fprop_ok(int Cin, int Cout) { return !fp32_mode() && shape_fprop_ok(Cin, Cout); }
bool tensor_wgrad_ok(int Cin, int Cout) { return !fp32_mode() && shape_wgrad_ok(Cin, Cout); }

// generic convolution forward, KS = 1 or 3
int conv_forward(const float* x, const float* weight, const float* bias, float* out, int B, int Cin, int Cout, int H,
                 int W, int KS) {
    cudaStream_t st = ub_layer_stream();
    const int ntaps = KS * KS;
    if (B < 1 || Cin < 1 || Cout < 1 || H < 1 || W < 1) {
        fail("conv forward: bad shape");
        return UB_ERR_SHAPE;
    }
    if (!tensor_fprop_ok(Cin, Cout)) {
        f32::conv_direct_fwd(x, weight, bias, out, B, Cin, Cout, H, W, KS, st);
        return finish(1);
    }
    std::lock_guard<std::mutex> lk(g_ws.mu);
    const size_t npix = size_t(B) * H * W;
    bf16* xb = (bf16*)g_ws.get(0, npix * Cin * 2);
    bf16* wp = (bf16*)g_ws.get(1, size_t(ntaps) * Cout * Cin * 2);
    if (!xb || !wp) {
        fail("workspace allocation failed");
        return UB_ERR_CUDA;
    }
    f32::nchw_to_nhwc_bf16(x, B, Cin, H * W, xb, st);
    if (pack_one(weight, wp, nullptr, Cout, Cin, ntaps, st)) return UB_ERR_CUDA;
    ConvSegDesc seg{xb, Cin, Cin, wp, ntaps};
    ConvEpilogue ep;
    ep.bias = bias, ep.out = out, ep.out_mode = OUT_NCHW_F32;
    IgemmConvParams p;
    int r = igemm_conv_plan(&p, &seg, 1, B, H, W, Cout, ep);
    if (r) {
        fail("conv forward: igemm plan failed (%d)", r);
        return UB_ERR_SHAPE;
    }
    igemm_conv_launch(p, st);
    return finish(3);
}

int conv_backward(const float* dout, const float* x, const float* weight, float* dx, float* dweight, float* dbias,
                  int B, int Cin, int Cout, int H, int W, int KS) {
    cudaStream_t st = ub_layer_stream();
    const int ntaps = KS * KS;
    const size_t npix = size_t(B) * H * W;
    std::lock_guard<std::mutex> lk(g_ws.mu);
    int launches = 0;
    const bool dgrad_tc = dx && tensor_fprop_ok(Cout, Cin);   // GEMM N = Cin, K = Cout
    const bool wgrad_tc = dweight && tensor_wgrad_ok(Cin, Cout);
    bf16 *dyb = nullptr, *xb = nullptr;
    if (dgrad_tc || wgrad_tc) {
        dyb = (bf16*)g_ws.get(2, npix * Cout * 2);
        if (!dyb) return UB_ERR_CUDA;
        f32::nchw_to_nhwc_bf16(dout, B, Cout, H * W, dyb, st);
        launches++;
    }
    if (dx) {
        if (dgrad_tc) {
            bf16* wd = (bf16*)g_ws.get(1, size_t(ntaps) * Cout * Cin * 2);
            if (!wd || pack_one(weight, nullptr, wd, Cout, Cin, ntaps, st)) return UB_ERR_CUDA;
            ConvSegDesc seg{dyb, Cout, Cout, wd, ntaps};
            ConvEpilogue ep;
            ep.out = dx, ep.out_mode = OUT_NCHW_F32;
            IgemmConvParams p;
            int r = igemm_conv_plan(&p, &seg, 1, B, H, W, Cin, ep);
            if (r) {
                fail("conv backward: dgrad plan failed (%d)", r);
                return UB_ERR_SHAPE;
            }
            igemm_conv_launch(p, st);
            launches += 2;
        } else {
            f32::conv_direct_dgrad(dout, weight, dx, B, Cin, Cout, H, W, KS, st);
            launches++;
        }
    }
    if (dweight) {
        if (wgrad_tc) {
            xb = (bf16*)g_ws.get(0, npix * Cin * 2);
            const size_t cap = size_t(16) << 20;  // floats
            float* partial = (float*)g_ws.get(3, cap * sizeof(float));
            if (!xb || !partial) return UB_ERR_CUDA;
            f32::nchw_to_nhwc_bf16(x, B, Cin, H * W, xb, st);
            IgemmWgradParams p;
            int r = igemm_wgrad_plan(&p, dyb, Cout, xb, Cin, B, H, W, Cin, Cout, ntaps, partial, cap, sm_count());
            if (r) {
                fail("conv backward: wgrad plan failed (%d)", r);
                return UB_ERR_SHAPE;
            }
            igemm_wgrad_launch(p, st);
            igemm_wgrad_reduce(p, dweight, st);
            launches += 3;
            if (dbias) f32::nchw_chansum(dout, B, Cout, size_t(H) * W, dbias, st), launches++;
        } else {
            f32::conv_direct_wgrad(dout, x, dweight, dbias, B, Cin, Cout, H, W, KS, st);
            launches += 2;
        }
    } else if (dbias) {
        f32::nchw_chansum(dout, B, Cout, size_t(H) * W, dbias, st), launches++;
    }
    return finish(launches);
}

}  // namespace

extern "C" {
int ub_set_layer_precision(int mode) {
    const int prev = fp32_mode() ? UB_PRECISION_FP32 : UB_PRECISION_BF16;
    g_precision = mode == UB_PRECISION_FP32 ? UB_PRECISION_FP32 : UB_PRECISION_BF16;
    return prev;
}

int ub_conv2d_k3_forward3(const float* x, const float* weight, const float* bias, float* out, int B, int C_in,
                          int C_out, int H, int W) {
    return conv_forward(x, weight, bias, out, B, C_in, C_out, H, W, 3);
}
int ub_conv2d_k3_forward2(const float* x, const float* weight, const float* bias, float* out, int B, int C_in,
                          int C_out, int H, int W) {
    return conv_forward(x, weight, bias, out, B, C_in, C_out, H, W, 3);
}
int ub_conv2d_k3_backward2(const float* dout, const float* x, const float* weight, float* /*dweight_buf*/,
                           float* /*dbias_buf*/, float* dx, float* dweight, float* dbias, int B, int C_in, int C_out,
                           int H, int W) {
    return conv_backward(dout, x, weight, dx, dweight, dbias, B, C_in, C_out, H, W, 3);
}
int ub_conv2d_k3_backward1(const float* dout, const float* x, const float* weight, float* dx, float* dweight,
                           float* dbias, int B, int C_in, int C_out, int H, int W) {
    return conv_backward(dout, x, weight, dx, dweight, dbias, B, C_in, C_out, H, W, 3);
}
int ub_conv2d_k1_forward2(const float* x, const float* weight, const float* bias, float* out, int B, int C_in, int H,
                          int W, int C_out) {
    return conv_forward(x, weight, bias, out, B, C_in, C_out, H, W, 1);
}
int ub_conv2d_k1_forward1(float* out, const float* x, const float* weight, const float* bias, int B, int C_in, int H,
                          int W, int C_out) {
    return conv_forward(x, weight, bias, out, B, C_in, C_out, H, W, 1);
}
int ub_conv2d_k1_backward1(const float* dout, const float* x, const float* weight, float* dx, float* dweight,
                           float* dbias, int B, int C_in, int C_out, int H, int W) {
    return conv_backward(dout, x, weight, dx, dweight, dbias, B, C_in, C_out, H, W, 1);
}

// ---- linear: out (N,OC) = inp (N,C) . W(OC,C)^T + b.  A (N,C) row-major matrix is an NHWC image with W = N.
int ub_matmul_forward2(float* out, const float* inp, const float* weight, const float* bias, int N, int C, int OC) {
    cudaStream_t st = ub_layer_stream();
    if (N < 128 || !tensor_fprop_ok(C, OC)) {  // tiny / odd problems: exact fp32, latency bound anyway
        f32::linear_fwd(out, inp, weight, bias, N, C, OC, st);
        return finish(1);
    }
    std::lock_guard<std::mutex> lk(g_ws.mu);
    bf16* xb = (bf16*)g_ws.get(0, size_t(N) * C * 2);
    bf16* wp = (bf16*)g_ws.get(1, size_t(OC) * C * 2);
    if (!xb || !wp) return UB_ERR_CUDA;
    f32::cast_bf16(inp, size_t(N) * C, xb, st);
    f32::cast_bf16(weight, size_t(OC) * C, wp, st);  // (OC, C) is already the K-major fprop pack of a 1-tap conv
    ConvSegDesc seg{xb, C, C, wp, 1};
    ConvEpilogue ep;
    ep.bias = bias, ep.out = out, ep.out_mode = OUT_NHWC_F32;
    IgemmConvParams p;
    int r = igemm_conv_plan(&p, &seg, 1, 1, 1, N, OC, ep);
    if (r) {
        fail("matmul_forward2: igemm plan failed (%d)", r);
        return UB_ERR_SHAPE;
    }
    igemm_conv_launch(p, st);
    return finish(3);
}
int ub_matmul_backward1(float* dinp, float* dweight, float* dbias, const float* dout, const float* inp,
                        const float* weight, int N, int C, int OC) {
    cudaStream_t st = ub_layer_stream();
    if (N < 128 || !tensor_fprop_ok(OC, C) || !tensor_wgrad_ok(C, OC)) {
        f32::linear_bwd(dinp, dweight, dbias, dout, inp, weight, N, C, OC, st);
        return finish(2);
    }
    std::lock_guard<std::mutex> lk(g_ws.mu);
    bf16* dyb = (bf16*)g_ws.get(2, size_t(N) * OC * 2);
    bf16* xb = (bf16*)g_ws.get(0, size_t(N) * C * 2);
    bf16* wd = (bf16*)g_ws.get(1, size_t(OC) * C * 2);
    const size_t cap = size_t(16) << 20;
    float* partial = (float*)g_ws.get(3, cap * sizeof(float));
    if (!dyb || !xb || !wd || !partial) return UB_ERR_CUDA;
    f32::cast_bf16(dout, size_t(N) * OC, dyb, st);
    f32::cast_bf16(inp, size_t(N) * C, xb, st);
    int launches = 2;
    if (dinp) {
        if (pack_one(weight, nullptr, wd, OC, C, 1, st)) return UB_ERR_CUDA;
        ConvSegDesc seg{dyb, OC, OC, wd, 1};
        ConvEpilogue ep;
        ep.out = dinp, ep.out_mode = OUT_NHWC_F32;
        IgemmConvParams p;
        int r = igemm_conv_plan(&p, &seg, 1, 1, 1, N, C, ep);
        if (r) {
            fail("matmul_backward1: dgrad plan failed (%d)", r);
            return UB_ERR_SHAPE;
        }
        igemm_conv_launch(p, st);
        launches += 2;
    }
    IgemmWgradParams p;
    int r = igemm_wgrad_plan(&p, dyb, OC, xb, C, 1, 1, N, C, OC, 1, partial, cap, sm_count());
    if (r) {
        fail("matmul_backward1: wgrad plan failed (%d)", r);
        return UB_ERR_SHAPE;
    }
    igemm_wgrad_launch(p, st);
    igemm_wgrad_reduce(p, dweight, st);
    if (dbias) f32::rows_colsum(dout, N, OC, dbias, st);
    return finish(launches + 3);
}

// ---- memory-bound operators (exact fp32, reference layouts)
int ub_groupnorm_forward(const float* x, const float* weight, const float* bias, float* out, float* mean,
                         float* rstd, int B, int C, int H, int W, int n_groups) {
    if (n_groups < 1 || C % n_groups) {
        fail("groupnorm: C %% n_groups != 0");
        return UB_ERR_SHAPE;
    }
    f32::groupnorm_fwd(x, weight, bias, out, mean, rstd, B, C, H * W, n_groups, ub_layer_stream());
    return finish(1);
}
int ub_groupnorm_backward(const float* dout, const float* x, const float* mean, const float* rstd,
                          const float* weight, float* dx, float* dweight, float* dbias, int B, int C, int H, int W,
                          int n_groups) {
    if (n_groups < 1 || C % n_groups) {
        fail("groupnorm: C %% n_groups != 0");
        return UB_ERR_SHAPE;
    }
    f32::groupnorm_bwd(dout, x, mean, rstd, weight, dx, dweight, dbias, B, C, H * W, n_groups, ub_layer_stream());
    return finish(1);
}
int ub_silu_forward(const float* x, float* out, int N) {
    f32::silu_fwd(x, out, size_t(N), ub_layer_stream());
    return finish(1);
}
int ub_silu_backward(const float* dout, const float* x, float* dx, int N) {
    f32::silu_bwd(dout, x, dx, size_t(N), ub_layer_stream());
    return finish(1);
}
int ub_add_forward(const float* a, const float* b, float* out, int N) {
    f32::add(a, b, out, size_t(N), ub_layer_stream());
    return finish(1);
}
int ub_add_inplace_forward(const float* a, float* b, int N) {
    f32::add(a, b, b, size_t(N), ub_layer_stream());
    return finish(1);
}
int ub_upsample_forward1(float* out, const float* x, int B, int C, int H, int W) {
    f32::upsample_fwd(out, x, size_t(B) * C, H, W, ub_layer_stream());
    return finish(1);
}
int ub_upsample_backward1(float* dx, const float* dout, int B, int C, int H, int W) {
    f32::upsample_bwd(dx, dout, size_t(B) * C, H, W, ub_layer_stream());
    return finish(1);
}
int ub_avgpool_2d_forward1(float* out, const float* x, int B, int C, int H, int W) {
    if ((H | W) & 1) {
        fail("avgpool: H and W must be even");
        return UB_ERR_SHAPE;
    }
    f32::avgpool_fwd(out, x, size_t(B) * C, H, W, ub_layer_stream());
    return finish(1);
}
int ub_avgpool_2d_backward1(const float* dout, float* dx, int B, int C, int H, int W) {
    if ((H | W) & 1) {
        fail("avgpool: H and W must be even");
        return UB_ERR_SHAPE;
    }
    f32::avgpool_bwd(dout, dx, size_t(B) * C, H, W, ub_layer_stream());
    return finish(1);
}
int ub_concat_channel_forward(const float* x1, const float* x2, float* out, int B, int C1, int C2, int H, int W) {
    f32::concat_fwd(x1, x2, out, B, C1, C2, H * W, ub_layer_stream());
    return finish(1);
}
int ub_concat_channel_backward(const float* dout, float* dx1, float* dx2, int B, int C1, int C2, int H, int W) {
    f32::concat_bwd(dout, dx1, dx2, B, C1, C2, H * W, ub_layer_stream());
    return finish(1);
}
int ub_broadcast_last_dims_forward(const float* x, float* out, int N, int H, int W) {
    f32::broadcast_fwd(x, out, size_t(N), H * W, ub_layer_stream());
    return finish(1);
}
int ub_broadcast_last_dims_backward(const float* dout, float* dx, int N, int H, int W) {
    f32::broadcast_bwd(dout, dx, size_t(N), H * W, ub_layer_stream());
    return finish(1);
}
int ub_mse_forward(const float* inp, const float* y, float* loss, int N) {
    f32::mse_fwd(inp, y, loss, size_t(N), ub_layer_stream());
    return finish(1);
}
int ub_mse_backward(const float* inp, const float* y, float* dinp, int N) {
    f32::mse_bwd(inp, y, dinp, size_t(N), ub_layer_stream());
    return finish(1);
}
int ub_get_timestep_embeddings(const float* timesteps, float* out, int B, int dim, int max_period) {
    if (dim & 1) {
        fail("timestep embedding: dim must be even");
        return UB_ERR_SHAPE;
    }
    timestep_embedding(timesteps, B, dim, max_period, out, ub_layer_stream());
    return finish(1);
}
int ub_attention_forward1(float* out, float* qkvr, float* preatt, float* att, const float* inp, int B, int T, int C,
                          int NH) {
    if (NH < 1 || C % NH) {
        fail("attention: C %% NH != 0");
        return UB_ERR_SHAPE;
    }
    f32::attention_fwd(out, qkvr, preatt, att, inp, B, T, C, NH, ub_layer_stream());
    return finish(3);
}
int ub_attention_backward(float* dinp, float* dqkvr, float* dpreatt, float* datt, float* /*scratch*/,
                          const float* dout, const float* qkvr, const float* att, int B, int T, int C, int NH) {
    if (NH < 1 || C % NH) {
        fail("attention: C %% NH != 0");
        return UB_ERR_SHAPE;
    }
    f32::attention_bwd(dinp, dqkvr, dpreatt, datt, dout, qkvr, att, B, T, C, NH, ub_layer_stream());
    return finish(3);
}

// ---- native-layout entry points (NHWC bf16)
int ub_nchw_to_nhwc_bf16(const float* x, void* y, int B, int C, int H, int W) {
    f32::nchw_to_nhwc_bf16(x, B, C, H * W, (bf16*)y, ub_layer_stream());
    return finish(1);
}
int ub_pack_conv_weight(const float* weight, void* wf, void* wd, int C_in, int C_out, int ksize) {
    std::lock_guard<std::mutex> lk(g_ws.mu);
    if (pack_one(weight, (bf16*)wf, (bf16*)wd, C_out, C_in, ksize * ksize, ub_layer_stream())) return UB_ERR_CUDA;
    return finish(1);
}
int ub_groupnorm_nhwc_forward(const void* x, const float* weight, const float* bias, void* y, float* chsum, int B, int H,
                              int W, int C, int n_groups, int silu, int impl) {
    if (n_groups < 1 || C % n_groups || C % 8) {
        fail("groupnorm_nhwc: needs C %% n_groups == 0 and C %% 8 == 0");
        return UB_ERR_SHAPE;
    }
    cudaStream_t st = ub_layer_stream();
    const int HW = H * W;
    if (impl == 0 && gn_slab_supported(B, HW, C, n_groups, false)) {
        if (gn_slab_fwd((const bf16*)x, C, weight, bias, B, HW, C, n_groups, silu, (bf16*)y, C, chsum, st)) {
            fail("groupnorm_nhwc_forward: slab launch rejected (alignment)");
            return UB_ERR_SHAPE;
        }
        return finish(1);
    }
    cudaMemsetAsync(chsum, 0, size_t(B) * C * 2 * sizeof(float), st);
    gn_stats((const bf16*)x, C, B, HW, C, chsum, st);
    gn_apply((const bf16*)x, C, chsum, weight, bias, B, HW, C, n_groups, silu, (bf16*)y, C, nullptr, st);
    return finish(2);
}
int ub_groupnorm_nhwc_backward(const void* x, const void* dy, const float* chsum, const float* weight, const float* bias,
                               const void* add_in, void* dx, float* dweight, float* dbias, float* scratch, int B, int H,
                               int W, int C, int n_groups, int silu, int impl) {
    if (n_groups < 1 || C % n_groups || C % 8) {
        fail("groupnorm_nhwc: needs C %% n_groups == 0 and C %% 8 == 0");
        return UB_ERR_SHAPE;
    }
    cudaStream_t st = ub_layer_stream();
    const int HW = H * W;
    if (impl == 0 && gn_slab_supported(B, HW, C, n_groups, true)) {
        if (gn_slab_bwd((const bf16*)x, C, (const bf16*)dy, C, chsum, weight, bias, B, HW, C, n_groups, silu,
                        (const bf16*)add_in, C, (bf16*)dx, C, dweight, dbias, nullptr, st)) {
            fail("groupnorm_nhwc_backward: slab launch rejected (alignment)");
            return UB_ERR_SHAPE;
        }
        return finish(1);
    }
    if (!scratch) {
        fail("groupnorm_nhwc_backward: the two-pass path needs scratch [B][C][2]");
        return UB_ERR_SHAPE;
    }
    cudaMemsetAsync(scratch, 0, size_t(B) * C * 2 * sizeof(float), st);
    gn_bwd_stats((const bf16*)x, C, (const bf16*)dy, C, chsum, weight, bias, B, HW, C, n_groups, silu, scratch, st);
    gn_bwd_apply((const bf16*)x, C, (const bf16*)dy, C, chsum, scratch, weight, bias, B, HW, C, n_groups, silu,
                 (const bf16*)add_in, C, (bf16*)dx, C, dweight, dbias, nullptr, st);
    return finish(2);
}
int ub_groupnorm_nhwc_backward_apply(const void* x, const void* dz, const float* chsum, const float* S,
                                     const float* weight, const float* bias, const void* add_in, void* dx,
                                     float* dweight, float* dbias, int B, int H, int W, int C, int n_groups, int silu) {
    if (n_groups < 1 || C % n_groups || C % 8) {
        fail("groupnorm_nhwc: needs C %% n_groups == 0 and C %% 8 == 0");
        return UB_ERR_SHAPE;
    }
    gn_bwd_apply((const bf16*)x, C, (const bf16*)dz, C, chsum, S, weight, bias, B, H * W, C, n_groups, silu ? 2 : 0,
                 (const bf16*)add_in, C, (bf16*)dx, C, dweight, dbias, nullptr, ub_layer_stream());
    return finish(1);
}
int ub_conv2d_nhwc_forward(const void* x, const void* wf, const float* bias, void* out, int B, int H, int W, int C_in,
                           int C_out, int ksize) {
    if (!shape_fprop_ok(C_in, C_out)) {
        fail("conv2d_nhwc_forward needs C_in %% 8 == 0 and C_out %% 16 == 0");
        return UB_ERR_SHAPE;
    }
    ConvSegDesc seg{(const bf16*)x, C_in, C_in, (const bf16*)wf, ksize * ksize};
    ConvEpilogue ep;
    ep.bias = bias, ep.out = out, ep.out_mode = OUT_NHWC_BF16;
    IgemmConvParams p;
    int r = igemm_conv_plan(&p, &seg, 1, B, H, W, C_out, ep);
    if (r) {
        fail("conv2d_nhwc_forward: plan failed (%d)", r);
        return UB_ERR_SHAPE;
    }
    igemm_conv_launch(p, ub_layer_stream());
    return finish(1);
}
int ub_conv2d_nhwc_dgrad(const void* dout, const void* wd, void* dx, int B, int H, int W, int C_in, int C_out,
                         int ksize) {
    if (!shape_fprop_ok(C_out, C_in)) {
        fail("conv2d_nhwc_dgrad needs C_out %% 8 == 0 and C_in %% 16 == 0");
        return UB_ERR_SHAPE;
    }
    ConvSegDesc seg{(const bf16*)dout, C_out, C_out, (const bf16*)wd, ksize * ksize};
    ConvEpilogue ep;
    ep.out = dx, ep.out_mode = OUT_NHWC_BF16;
    IgemmConvParams p;
    int r = igemm_conv_plan(&p, &seg, 1, B, H, W, C_in, ep);
    if (r) {
        fail("conv2d_nhwc_dgrad: plan failed (%d)", r);
        return UB_ERR_SHAPE;
    }
    igemm_conv_launch(p, ub_layer_stream());
    return finish(1);
}
int ub_conv2d_nhwc_wgrad(const void* dout, const void* x, float* dweight, float* dbias, int B, int H, int W, int C_in,
                         int C_out, int ksize) {
    if (!shape_wgrad_ok(C_in, C_out)) {
        fail("conv2d_nhwc_wgrad needs C_in %% 64 == 0 and C_out %% 64 == 0");
        return UB_ERR_SHAPE;
    }
    cudaStream_t st = ub_layer_stream();
    std::lock_guard<std::mutex> lk(g_ws.mu);
    const size_t cap = size_t(16) << 20;
    float* partial = (float*)g_ws.get(3, cap * sizeof(float));
    if (!partial) return UB_ERR_CUDA;
    IgemmWgradParams p;
    int r = igemm_wgrad_plan(&p, (const bf16*)dout, C_out, (const bf16*)x, C_in, B, H, W, C_in, C_out, ksize * ksize,
                             partial, cap, sm_count());
    if (r) {
        fail("conv2d_nhwc_wgrad: plan failed (%d)", r);
        return UB_ERR_SHAPE;
    }
    igemm_wgrad_launch(p, st);
    igemm_wgrad_reduce(p, dweight, st);
    int launches = 2;
    if (dbias) {
        cudaMemsetAsync(dbias, 0, size_t(C_out) * sizeof(float), st);
        colsum((const bf16*)dout, C_out, size_t(B) * H * W, C_out, dbias, nullptr, st);
        launches++;
    }
    return finish(launches);
}

int ub_conv2d_nhwc_fused(const UbConvSeg* segs, int nseg, int B, int H, int W, int C_out, const UbConvEpilogue* ep,
                         int kernel, UbConvPlanInfo* info) {
    UbConvPlanInfo inf{};
    inf.kernel = kernel;
    if (info) *info = inf;
    if (!segs || nseg < 1 || nseg > 2 || !ep || (kernel != 0 && kernel != 1) || B < 1 || H < 1 || W < 1) {
        fail("conv2d_nhwc_fused: bad arguments (nseg 1 or 2, kernel 0 or 1, epilogue required)");
        return UB_ERR_SHAPE;
    }
    ConvSegDesc sd[2];
    for (int s = 0; s < nseg; ++s) {
        if (segs[s].ksize != 1 && segs[s].ksize != 3) {
            fail("conv2d_nhwc_fused: ksize must be 1 or 3");
            return UB_ERR_SHAPE;
        }
        sd[s] = ConvSegDesc{(const bf16*)segs[s].x_bf16, segs[s].C_in, segs[s].ldx ? segs[s].ldx : segs[s].C_in,
                            (const bf16*)segs[s].w_bf16, segs[s].ksize * segs[s].ksize};
    }
    ConvEpilogue e;
    e.bias = ep->bias, e.bias2 = ep->bias2, e.rowvec = ep->rowvec;
    e.residual = (const bf16*)ep->residual_bf16, e.ldr = ep->ldr;
    e.out = ep->out, e.ldo = ep->ldo, e.out_mode = ep->out_mode;
    e.stats = ep->stats;
    e.gn_x = (const bf16*)ep->gn_x_bf16, e.gn_ldx = ep->gn_ldx ? ep->gn_ldx : C_out, e.gn_chsum = ep->gn_chsum;
    e.gn_gamma = ep->gn_gamma, e.gn_beta = ep->gn_beta, e.gn_S = ep->gn_S;
    e.gn_silu = ep->gn_silu, e.gn_groups = ep->gn_groups;
    if (e.out_mode < OUT_NHWC_BF16 || e.out_mode > OUT_NHWC_F32) {
        fail("conv2d_nhwc_fused: out_mode must be 0, 1 or 2");
        return UB_ERR_SHAPE;
    }
    cudaStream_t st = ub_layer_stream();
    if (kernel == 0) {
        IgemmConvParams p;
        const int r = igemm_conv_plan(&p, sd, nseg, B, H, W, C_out, e);
        inf.BN = p.BN, inf.nacc = p.nacc, inf.ms = p.ms, inf.stages = p.stages;
        inf.TW = p.TW, inf.TH = p.TH, inf.TB = p.TB;
        inf.grid = p.tiles_w * p.tiles_h * p.tiles_b * (p.BN ? C_out / p.BN : 0);
        if (info) *info = inf;
        if (r) {
            fail("conv2d_nhwc_fused: basic-kernel plan failed (%d)", r);
            return UB_ERR_SHAPE;
        }
        igemm_conv_launch(p, st);
    } else {
        if (!igemm_rows_eligible(B, H, W, C_out)) {
            fail("conv2d_nhwc_fused: the row-tile kernel needs W in {16, 32, 64, 128}, H >= 256 / W, C_out %% 16 == 0");
            return UB_ERR_SHAPE;
        }
        IgemmRowsParams p;
        const int r = igemm_rows_plan(&p, sd, nseg, B, H, W, C_out, e, sm_count());
        inf.BN = p.BN, inf.stages = p.a_stages, inf.w_resident = p.w_resident;
        inf.TW = W, inf.TH = p.TH, inf.TB = 1, inf.grid = p.grid;
        if (info) *info = inf;
        if (r) {
            fail("conv2d_nhwc_fused: row-tile plan failed (%d)", r);
            return UB_ERR_SHAPE;
        }
        igemm_rows_launch(p, st);
    }
    return finish(1);
}

int ub_conv2d_nhwc_wgrad_acc(const void* dout, int lddy, const void* x, int ldx, float* dweight, float* dbias,
                             float* dbias2, int B, int H, int W, int C_in, int C_out, int ksize, int* colmode_out,
                             int* nsplit_out) {
    if (!shape_wgrad_ok(C_in, C_out) || (ksize != 1 && ksize != 3) || !dweight || (dbias2 && !dbias)) {
        fail("conv2d_nhwc_wgrad_acc needs C_in %% 64 == 0, C_out %% 64 == 0, ksize 1 or 3, dweight, and dbias with dbias2");
        return UB_ERR_SHAPE;
    }
    const int ntaps = ksize * ksize;
    cudaStream_t st = ub_layer_stream();
    std::lock_guard<std::mutex> lk(g_ws.mu);
    float* acc = dweight;  // 1x1: [C_out][C_in] is the final layout, the kernel adds into it
    WgradFinalizeEntry* tab = nullptr;
    int launches = 1;
    if (ntaps == 9) {
        // [9][C_out][C_in] accumulator in workspace slot 4: zeroed when (re)allocated, re-zeroed by every finalize
        static void* zeroed = nullptr;
        static size_t zeroed_cap = 0;
        const size_t bytes = size_t(9) * C_out * C_in * sizeof(float);
        acc = (float*)g_ws.get(4, bytes);
        tab = (WgradFinalizeEntry*)g_ws.get(5, sizeof(WgradFinalizeEntry));
        if (!acc || !tab) {
            fail("workspace allocation failed");
            return UB_ERR_CUDA;
        }
        if (acc != zeroed || g_ws.cap[4] != zeroed_cap) {
            if (cudaMemsetAsync(acc, 0, g_ws.cap[4], st) != cudaSuccess) return finish(0);
            zeroed = acc, zeroed_cap = g_ws.cap[4];
        }
        const WgradFinalizeEntry e{acc, dweight, C_out, C_in};
        if (cudaMemcpyAsync(tab, &e, sizeof e, cudaMemcpyHostToDevice, st) != cudaSuccess) return finish(0);
    }
    IgemmWgradParams p;
    const int r = igemm_wgrad_plan_acc(&p, (const bf16*)dout, lddy ? lddy : C_out, (const bf16*)x, ldx ? ldx : C_in, B,
                                       H, W, C_in, C_out, ntaps, acc, dbias, dbias2, sm_count());
    if (colmode_out) *colmode_out = p.colmode;
    if (nsplit_out) *nsplit_out = p.nsplit;
    if (r) {
        fail("conv2d_nhwc_wgrad_acc: plan failed (%d)", r);
        return UB_ERR_SHAPE;
    }
    igemm_wgrad_launch(p, st);
    if (tab) igemm_wgrad_finalize(tab, 1, size_t(C_out) * C_in, st), launches++;
    return finish(launches);
}

}  // extern "C"

extern "C" {
// ---- attention core, native layout
// head size C / NH (32 or 64) if impl can run the shape, else 0 with the reason set
static int attention_shape_check(int C, int NH, int T, int impl) {
    const int HS = NH < 1 ? 0 : (C == NH * 32 ? 32 : (C == NH * 64 ? 64 : 0));
    if (!HS) {
        fail("attention_nhwc: head size must be 32 or 64 (C == NH * 32 or C == NH * 64)");
        return 0;
    }
    if (impl == 0 && !attn_tc_supported(T, NH, HS)) {
        fail("attention_nhwc: the tcgen05 kernels need T in {16,32,64,128,256} and, at head size 32, an even NH");
        return 0;
    }
    return HS;
}

int ub_attention_nhwc_forward(const void* qkv, void* out, float* lse, int B, int T, int C, int NH, int impl) {
    const int HS = attention_shape_check(C, NH, T, impl);
    if (!HS) return UB_ERR_SHAPE;
    if (impl == 0) {
        AttnTcParams p;
        int r = attn_tc_plan(&p, (const bf16*)qkv, 3 * C, B, T, NH, HS, (bf16*)out, C, lse, nullptr, 0, nullptr, 0,
                             nullptr);
        if (r) {
            fail("attn_tc_plan failed (%d)", r);
            return UB_ERR_SHAPE;
        }
        attn_tc_fwd(p, ub_layer_stream());
    } else {
        attn_fwd((const bf16*)qkv, 3 * C, B, T, NH, HS, (bf16*)out, C, lse, ub_layer_stream());
    }
    return finish(1);
}
int ub_attention_nhwc_backward(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv,
                               float* dsum, int B, int T, int C, int NH, int impl) {
    const int HS = attention_shape_check(C, NH, T, impl);
    if (!HS) return UB_ERR_SHAPE;
    if (impl == 0) {
        AttnTcParams p;
        int r = attn_tc_plan(&p, (const bf16*)qkv, 3 * C, B, T, NH, HS, (bf16*)const_cast<void*>(out), C,
                             const_cast<float*>(lse), (const bf16*)dout, C, (bf16*)dqkv, 3 * C, dsum);
        if (r) {
            fail("attn_tc_plan failed (%d)", r);
            return UB_ERR_SHAPE;
        }
        attn_tc_bwd(p, ub_layer_stream());
    } else {
        attn_bwd((const bf16*)qkv, 3 * C, (const bf16*)out, C, (const bf16*)dout, C, lse, B, T, NH, HS, (bf16*)dqkv,
                 3 * C, dsum, ub_layer_stream());
    }
    return finish(2);
}

// ---- composite blocks: the op sequence and buffer roles are the reference's contract (dev/resblock.cu:24-200,
//      dev/attention_block.cu:64-108); each step is one of the operators above.
#define UB_STEP(call)        \
    do {                     \
        int rc_ = (call);    \
        if (rc_) return rc_; \
    } while (0)

static int resample(float* out, const float* x, int B, int C, int H, int W, int up, int down) {
    if (up) return ub_upsample_forward1(out, x, B, C, H, W);
    if (down) return ub_avgpool_2d_forward1(out, x, B, C, H, W);
    if (cudaMemcpyAsync(out, x, size_t(B) * C * H * W * sizeof(float), cudaMemcpyDeviceToDevice, ub_layer_stream()) !=
        cudaSuccess) {
        fail("resblock: device copy failed");
        return UB_ERR_CUDA;
    }
    return UB_OK;
}
static int resample_bwd(const float* dout, float* dx, int B, int C, int H, int W, int up, int down) {
    if (up) return ub_upsample_backward1(dx, dout, B, C, H, W);
    if (down) return ub_avgpool_2d_backward1(dout, dx, B, C, H, W);
    if (cudaMemcpyAsync(dx, dout, size_t(B) * C * H * W * sizeof(float), cudaMemcpyDeviceToDevice, ub_layer_stream()) !=
        cudaSuccess) {
        fail("resblock: device copy failed");
        return UB_ERR_CUDA;
    }
    return UB_OK;
}

int ub_resblock_forward(int C, int C_emb, int C_out, int B, int H, int W, int up, int down, int G,
                        const UbResBlockParams* p, const UbResBlockActs* a) {
    if (up && down) {
        fail("resblock: up and down are exclusive");
        return UB_ERR_SHAPE;
    }
    const int Ho = up ? 2 * H : (down ? H / 2 : H), Wo = up ? 2 * W : (down ? W / 2 : W);
    const int n_in = B * C * H * W, n_out = B * C_out * Ho * Wo;
    // GroupNorm -> SiLU -> (resample) -> 3x3 conv
    UB_STEP(ub_groupnorm_forward(a->input, p->gn1_w, p->gn1_b, a->gn1, a->gn1_mean, a->gn1_rstd, B, C, H, W, G));
    UB_STEP(ub_silu_forward(a->gn1, a->silu1, n_in));
    UB_STEP(resample(a->ud_h, a->silu1, B, C, H, W, up, down));
    UB_STEP(resample(a->ud_x, a->input, B, C, H, W, up, down));
    UB_STEP(ub_conv2d_k3_forward3(a->ud_h, p->cv3_1_w, p->cv3_1_b, a->cv3_1, B, C, C_out, Ho, Wo));
    // time embedding: SiLU -> Linear -> broadcast over the pixels -> add
    UB_STEP(ub_silu_forward(a->emb, a->silu_emb, B * C_emb));
    UB_STEP(ub_matmul_forward2(a->l_emb, a->silu_emb, p->l_emb_w, p->l_emb_b, B, C_emb, C_out));
    UB_STEP(ub_broadcast_last_dims_forward(a->l_emb, a->broad_emb, B * C_out, Ho, Wo));
    UB_STEP(ub_add_forward(a->cv3_1, a->broad_emb, a->add1, n_out));
    // GroupNorm -> SiLU -> 3x3 conv
    UB_STEP(ub_groupnorm_forward(a->add1, p->gn2_w, p->gn2_b, a->gn2, a->gn2_mean, a->gn2_rstd, B, C_out, Ho, Wo, G));
    UB_STEP(ub_silu_forward(a->gn2, a->silu2, n_out));
    UB_STEP(ub_conv2d_k3_forward3(a->silu2, p->cv3_2_w, p->cv3_2_b, a->cv3_2, B, C_out, C_out, Ho, Wo));
    // residual, through a 1x1 conv when the channel count changes
    if (C_out == C) return ub_add_forward(a->cv3_2, a->ud_x, a->add2, n_out);
    UB_STEP(ub_conv2d_k1_forward2(a->ud_x, p->res_cv1_w, p->res_cv1_b, a->res_cv1, B, C, Ho, Wo, C_out));
    return ub_add_forward(a->cv3_2, a->res_cv1, a->add2, n_out);
}

int ub_resblock_backward(int C, int C_emb, int C_out, int B, int H, int W, int up, int down, int G,
                         const UbResBlockParams* p, const UbResBlockParams* g, const UbResBlockActs* a,
                         const UbResBlockBack* k) {
    if (up && down) {
        fail("resblock: up and down are exclusive");
        return UB_ERR_SHAPE;
    }
    const int Ho = up ? 2 * H : (down ? H / 2 : H), Wo = up ? 2 * W : (down ? W / 2 : W);
    const int n_in = B * C * H * W, n_out = B * C_out * Ho * Wo;
    // scratch, as the reference: the two last forward activations (C_out channels) and, once the skip conv has been
    // differentiated, ud_x (C channels at the output resolution)
    float *s1 = a->cv3_2, *s2 = a->add2, *sx = a->ud_x;
    const float* d_skip = k->dout;  // gradient of the residual branch at the output resolution
    if (C_out != C) {
        UB_STEP(ub_conv2d_k1_backward1(k->dout, a->ud_x, p->res_cv1_w, k->buf_BCHoWo, g->res_cv1_w, g->res_cv1_b, B, C,
                                       C_out, Ho, Wo));
        d_skip = k->buf_BCHoWo;
    }
    // conv2 <- SiLU <- GroupNorm2
    UB_STEP(ub_conv2d_k3_backward2(k->dout, a->silu2, p->cv3_2_w, nullptr, nullptr, s1, g->cv3_2_w, g->cv3_2_b, B, C_out,
                                   C_out, Ho, Wo));
    UB_STEP(ub_silu_backward(s1, a->gn2, s2, n_out));
    UB_STEP(ub_groupnorm_backward(s2, a->add1, a->gn2_mean, a->gn2_rstd, p->gn2_w, s1, g->gn2_w, g->gn2_b, B, C_out, Ho,
                                  Wo, G));
    // embedding branch: sum over pixels -> Linear backward -> SiLU backward
    UB_STEP(ub_broadcast_last_dims_backward(s1, a->l_emb, B * C_out, Ho, Wo));
    UB_STEP(ub_matmul_backward1(k->buf_BCemb, g->l_emb_w, g->l_emb_b, a->l_emb, a->silu_emb, p->l_emb_w, B, C_emb,
                                C_out));
    UB_STEP(ub_silu_backward(k->buf_BCemb, a->emb, k->demb, B * C_emb));
    // conv1 <- (resample) <- SiLU <- GroupNorm1, plus the residual branch
    UB_STEP(ub_conv2d_k3_backward2(s1, a->ud_h, p->cv3_1_w, nullptr, nullptr, sx, g->cv3_1_w, g->cv3_1_b, B, C, C_out, Ho,
                                   Wo));
    UB_STEP(resample_bwd(sx, k->buf1_BCHW, B, C, H, W, up, down));
    UB_STEP(resample_bwd(d_skip, k->buf2_BCHW, B, C, H, W, up, down));
    UB_STEP(ub_silu_backward(k->buf1_BCHW, a->gn1, a->silu1, n_in));
    UB_STEP(ub_groupnorm_backward(a->silu1, a->input, a->gn1_mean, a->gn1_rstd, p->gn1_w, k->buf1_BCHW, g->gn1_w, g->gn1_b,
                                  B, C, H, W, G));
    return ub_add_forward(k->buf1_BCHW, k->buf2_BCHW, k->dx, n_in);
}

int ub_attention_block_forward(int B, int C, int H, int W, int HS, int G, const UbAttentionParams* p,
                               const UbAttentionActs* a) {
    if (HS < 1 || C % HS) {
        fail("attention_block: C %% HS != 0");
        return UB_ERR_SHAPE;
    }
    const int T = H * W;
    UB_STEP(ub_groupnorm_forward(a->input, p->gn_w, p->gn_b, a->gn, a->gn_mean, a->gn_rstd, B, C, H, W, G));
    f32::permute_bchw_to_bhwc(a->gn, a->perm1, B, C, T, ub_layer_stream());
    UB_STEP(finish(1));
    UB_STEP(ub_matmul_forward2(a->qkv1, a->perm1, p->qkv_w, p->qkv_b, B * T, C, 3 * C));
    UB_STEP(ub_attention_forward1(a->att_out, a->qkv2, a->preatt, a->att, a->qkv1, B, T, C, C / HS));
    UB_STEP(ub_matmul_forward2(a->proj, a->att_out, p->proj_w, p->proj_b, B * T, C, C));
    f32::permute_bhwc_to_bchw(a->proj, a->perm2, B, C, T, ub_layer_stream());
    UB_STEP(finish(1));
    return ub_add_forward(a->input, a->perm2, a->add, B * C * T);
}

int ub_attention_block_backward(int B, int C, int H, int W, int HS, int G, const UbAttentionParams* p,
                                const UbAttentionActs* a, const UbAttentionBack* k, const UbAttentionParams* g) {
    if (HS < 1 || C % HS) {
        fail("attention_block: C %% HS != 0");
        return UB_ERR_SHAPE;
    }
    const int T = H * W;
    f32::permute_bchw_to_bhwc(k->dout, k->buf1_BCHW, B, C, T, ub_layer_stream());
    UB_STEP(finish(1));
    UB_STEP(ub_matmul_backward1(k->buf2_BCHW, g->proj_w, g->proj_b, k->buf1_BCHW, a->att_out, p->proj_w, B * T, C, C));
    UB_STEP(ub_attention_backward(k->buf_B3CHW, k->dqkvr, k->dpreatt, k->datt, k->buf1_BCHW, k->buf2_BCHW, a->qkv2, a->att,
                                  B, T, C, C / HS));
    UB_STEP(ub_matmul_backward1(k->buf1_BCHW, g->qkv_w, g->qkv_b, k->buf_B3CHW, a->perm1, p->qkv_w, B * T, C, 3 * C));
    f32::permute_bhwc_to_bchw(k->buf1_BCHW, k->buf2_BCHW, B, C, T, ub_layer_stream());
    UB_STEP(finish(1));
    UB_STEP(ub_groupnorm_backward(k->buf2_BCHW, a->input, a->gn_mean, a->gn_rstd, p->gn_w, k->buf1_BCHW, g->gn_w, g->gn_b,
                                  B, C, H, W, G));
    return ub_add_forward(k->buf1_BCHW, k->dout, k->dinp, B * C * T);
}
}  // extern "C"
