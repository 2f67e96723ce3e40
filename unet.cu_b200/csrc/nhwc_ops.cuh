// Memory-bound kernels of the internal (NHWC bf16) training path. All tensors are (ptr, ld) pairs:
// element (pixel p, channel c) lives at ptr[p * ld + c]; ld lets a kernel read/write a channel slice of a
// wider buffer (concat buffers, gradient-of-concat buffers) without a copy.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace ub {

typedef __nv_bfloat16 bf16;

// one-time kernel attribute setup (opt-in shared memory); call before graph capture
void nhwc_ops_init();

// ---- dropout behind a GroupNorm + SiLU (guided-diffusion's ResBlock out_layers: GroupNorm, SiLU, Dropout(p), conv; the
//      reference carries the option but has it commented out, dev/resblock.py:51,61, dev/unet.py:116,140).  The mask is
//      never stored: forward and backward regenerate it from Philox4x32-10 with counter = element index / 4 (NHWC order),
//      stream word = layer and key = (seed, step).  ctl (device) = {p as float bits, step, seed lo, seed hi}: written at
//      the start of every step (p = 0 for inference), so one captured graph serves all steps.  ctl == nullptr: no dropout.
struct DropArgs {
    const unsigned* ctl = nullptr;
    unsigned layer = 0;
};
void dropout_set_ctl(unsigned* ctl, float p, unsigned long long seed, const int* step_dev, cudaStream_t st);
// mask (0 / 1 bytes, NHWC element order) of `layer` for the (seed, step) recorded in ctl, with the drop probability p given here
void dropout_mask(const unsigned* ctl, float p, unsigned layer, size_t n, unsigned char* out, cudaStream_t st);

// ---- GroupNorm (+ optional SiLU), replaces groupnorm_forward/backward + silu_forward/backward
//      (/root/reference/train_unet.cu:1768-1991, :305-351).
// chsum: [B][C][2] fp32 per-(image, channel) sum and sum of squares (must be zero on entry to gn_stats).
void gn_stats(const bf16* x, int ldx, int B, int HW, int C, float* chsum, cudaStream_t st);
// y = act(gn(x)); also writes meanrstd[B][G][2] if non-null.
void gn_apply(const bf16* x, int ldx, const float* chsum, const float* gamma, const float* beta, int B, int HW, int C,
              int G, int silu, bf16* y, int ldy, float* meanrstd, cudaStream_t st, const float* ss = nullptr,
              DropArgs drop = DropArgs());
// ss (optional, use_scale_shift_norm, dev/resblock.py:243-247): [B][2C] fp32, per image [scale (C) | shift (C)];
// the normalised value becomes gn(x) * (1 + scale) + shift before the activation.  gn_bwd_stats / gn_bwd_apply take the
// same pointer; gn_bwd_apply (unfused, silu == 1) additionally writes dss [B][2C] = [dscale | dshift].
// Backward pass 1: S[B][C][2] = per-(image,channel) sums of dz and dz*xhat (must be zero on entry).
void gn_bwd_stats(const bf16* x, int ldx, const bf16* dy, int lddy, const float* chsum, const float* gamma,
                  const float* beta, int B, int HW, int C, int G, int silu, float* S, cudaStream_t st,
                  const float* ss = nullptr, DropArgs drop = DropArgs());
// Backward pass 2: dx = gn_bwd(dy) [+ add_in]; dgamma/dbeta += (atomic); colsum_out[B][C] += sum_pix dx (optional).
// silu: 0 = no activation, 1 = SiLU follows the norm (dy is dL/d silu(gn(x))), 2 = SiLU follows the norm and dy is
// already dL/d gn(x) (the dgrad conv that produced it applied silu' in its epilogue, see epilogue.cuh).
void gn_bwd_apply(const bf16* x, int ldx, const bf16* dy, int lddy, const float* chsum, const float* S,
                  const float* gamma, const float* beta, int B, int HW, int C, int G, int silu, const bf16* add_in,
                  int ldadd, bf16* dx, int lddx, float* dgamma, float* dbeta, float* colsum_out, cudaStream_t st,
                  const float* ss = nullptr, float* dss = nullptr, DropArgs drop = DropArgs());

// ---- single-pass GroupNorm (csrc/gn_slab.cu): statistics + normalisation (+SiLU) in ONE kernel, the slab (image, whole
//      groups of channels) held in registers in between: 1R + 1W forward, 2R (+1R) + 1W backward.  Return -1 when the
//      shape is not supported (channel count not a multiple of 16, slab too large): use the two-pass kernels above.
bool gn_slab_supported(int B, int HW, int C, int G, bool backward);
void gn_slab_init();  // opt-in shared memory attributes; called by nhwc_ops_init() (before graph capture)
// y = act(gn(x)); chsum[B][C][2] receives the per-(image, channel) sum / sum of squares (overwritten, for the backward)
int gn_slab_fwd(const bf16* x, int ldx, const float* gamma, const float* beta, int B, int HW, int C, int G, int silu,
                bf16* y, int ldy, float* chsum, cudaStream_t st);
// dx = gn_bwd(dy) [+ add_in]; dy = dL/d act(gn(x)) (silu: 0 identity, 1 SiLU); dgamma/dbeta += ; colsum_out[B][C] += sum_pix dx
int gn_slab_bwd(const bf16* x, int ldx, const bf16* dy, int lddy, const float* chsum, const float* gamma,
                const float* beta, int B, int HW, int C, int G, int silu, const bf16* add_in, int ldadd, bf16* dx,
                int lddx, float* dgamma, float* dbeta, float* colsum_out, cudaStream_t st);

// ---- data movement (replace avgpool/upsample/concat/add of train_unet.cu:187-627)
void avgpool2_fwd(const bf16* x, int ldx, int B, int H, int W, int C, bf16* y, int ldy, cudaStream_t st);
// dx (H x W) = dy (H/2 x W/2) / 4 [+ add_in]
void avgpool2_bwd(const bf16* dy, int lddy, int B, int H, int W, int C, const bf16* add_in, int ldadd, bf16* dx,
                  int lddx, cudaStream_t st);
// out[:, :C1] = up ? nearest_up2(a) : a ; out[:, C1:] = b.   (H, W) is the OUTPUT resolution.
// If cs_a and cs_b (GroupNorm statistics [B][C][2] of the two inputs) are given, cs_out receives the statistics of
// the concatenation.
void concat2(const bf16* a, int lda, int C1, int up, const bf16* b, int ldb, int C2, int B, int H, int W, bf16* out,
             int ldo, const float* cs_a, const float* cs_b, float* cs_out, cudaStream_t st);
// y (2H x 2W) = nearest x2 upsample of x (H x W); (H, W) is the INPUT resolution
void upsample2_fwd(const bf16* x, int ldx, int B, int H, int W, int C, bf16* y, int ldy, cudaStream_t st);
// dx (H/2 x W/2) = sum of the 4 children of dy (H x W)
void upsample2_bwd(const bf16* dy, int lddy, int B, int H, int W, int C, bf16* dx, int lddx, cudaStream_t st);
void add2(const bf16* a, int lda, const bf16* b, int ldb, size_t npix, int C, bf16* out, int ldo, cudaStream_t st);
// out[c] += sum_p x[p][c] (and out2[c] if non-null)   (fp32 atomics; outputs must be initialised)
void colsum(const bf16* x, int ldx, size_t npix, int C, float* out, float* out2, cudaStream_t st);

// ---- 3-channel convolutions (first / last layer of the U-Net) -- SIMT, negligible FLOPs
// conv_in: x NCHW fp32 (B,Cin<=4,H,W), w (Cout,Cin,3,3) fp32 -> y NHWC bf16.  Cin = 6 (super-resolution model): input
// channels 0-2 from x and 3-5 from x2, both (B,3,H,W) -- the row kernels only; x2 is null otherwise
void conv_in_fwd(const float* x, const float* x2, const float* w, const float* b, int B, int Cin, int Cout, int H,
                 int W, bf16* y, int ldy, cudaStream_t st);
// dW, db of conv_in from dy NHWC bf16 (overwrite); scratch >= blocks*(Cout*Cin*9 + Cout) floats; x2 as conv_in_fwd
void conv_in_wgrad(const float* x, const float* x2, const bf16* dy, int lddy, int B, int Cin, int Cout, int H, int W,
                   float* dw, float* db, float* scratch, size_t scratch_floats, cudaStream_t st);
// dx NCHW fp32 (B,Cin<=4,H,W) = conv_transpose(dh NHWC bf16 with Cout channels, w (Cout,Cw,3,3)) restricted to the first
// Cin input channels: dL/d(x_t) (Cw = Cin, or 2 Cin for a super-resolution model)
void conv_in_dgrad(const bf16* dh, int lddh, const float* w, int B, int Cin, int Cout, int H, int W, float* dx,
                   cudaStream_t st, int Cw);
// true when the row-per-warp conv_in kernels (forward and weight gradient) take Cs small channels at Cb big channels
// and width W -- what a super-resolution config (Cs = 6) needs, as no other kernel serves it
bool smallc_rows_fit(int Cs, int Cb, int W);
// conv_out: a NHWC bf16 (Cin = 64..), w (Cout<=4,Cin,3,3) -> out NCHW fp32
void conv_out_fwd(const bf16* a, int lda, const float* w, const float* b, int B, int Cin, int Cout, int H, int W,
                  float* out, cudaStream_t st);
// da NHWC bf16 = conv_transpose(dout NCHW fp32, w).  Cout = 6 (learned-variance head): dout holds the gradients of
// output channels 0-2 and dout2 those of 3-5, both (B,3,H,W) -- the row kernels only; dout2 is null otherwise
void conv_out_dgrad(const float* dout, const float* w, int B, int Cin, int Cout, int H, int W, bf16* da, int ldda,
                    cudaStream_t st, const float* dout2 = nullptr);
// dw, db (accumulated); dout2 as conv_out_dgrad
void conv_out_wgrad(const bf16* a, int lda, const float* dout, int B, int Cin, int Cout, int H, int W, float* dw,
                    float* db, float* scratch, size_t scratch_floats, cudaStream_t st, const float* dout2 = nullptr);
// true when the 6-output row kernel of the learned-variance head (conv_out_fwd_hybrid) takes Cin channels at width W
bool conv_out_rows_fit6(int Cin, int W);
// opt the 6-output row kernel into the dynamic shared memory conv_out_rows_fit6 allows, on the current device; on
// failure msg says why (a learned-variance trainer is not created then)
cudaError_t conv_out_rows_prepare6(char* msg, size_t msg_len);

// ---- loss (replaces mse_forward/backward, train_unet.cu:2981-3030): loss += mean((out-y)^2); dout = 2(out-y)/N
void conv_out_fwd_mse(const bf16* a, int lda, const float* w, const float* b, int B, int Cin, int Cout, int H, int W,
                      float* out, const float* target, float* loss, float* dout, float grad_scale, cudaStream_t st);
void mse_fwd_bwd(const float* out, const float* y, size_t N, float* loss, float* dout, float grad_scale,
                 cudaStream_t st);
// Learned-variance head (guided-diffusion's learn_sigma with the hybrid loss): what the epilogue of the 6-output conv
// reads beside the noise, and where it writes dL/dv.  coef holds 8 floats per timestep t < T, built in float64 and
// rounded: {sqrt(1/acp), sqrt(1/acp - 1), c1, c2, log beta, lpost, T/1000, 0}, c1 / c2 the posterior-mean coefficients
// of x0 / x_t and lpost the clipped log posterior variance.  x0 is the batch before random_flip (flips may be null).
struct HybridLoss {
    const float* xt;
    const float* x0;
    const float* t;  // (B) timesteps as floats
    const int* flips;
    const float* coef;
    float* dv;  // (B,3,H,W)
    int T;
};
// out (B,6,H,W) = conv3x3(a, w (6,Cin,3,3)) + b = [eps | v]; with noise: loss2[0] += mean (eps - noise)^2,
// loss2[1] += mean vb (bits, times T/1000); deps, hl.dv (B,3,H,W) = their gradients (eps only from the MSE, v only from
// vb) * grad_scale.  noise = null (inference): out only.  One launch; the shape must pass conv_out_rows_fit6 and
// conv_out_rows_prepare6 must have succeeded.
void conv_out_fwd_hybrid(const bf16* a, int lda, const float* w, const float* b, int B, int Cin, int H, int W,
                         float* out, const float* noise, float* loss2, float* deps, const HybridLoss& hl,
                         float grad_scale, cudaStream_t st);

}  // namespace ub
