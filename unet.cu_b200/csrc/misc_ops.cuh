// Remaining kernels of the internal training path: attention core, small fp32 linears (time-embedding MLP and
// the per-ResBlock embedding projections), diffusion noise / q-sample, weight packing, fused AdamW.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace ub {

typedef __nv_bfloat16 bf16;

// ---- attention core (replaces attention_forward1 / attention_backward, /root/reference/train_unet.cu:2553-2760)
// qkv: NHWC bf16 [B*T][ld], channel order [Q | K | V], each [NH][HS] (dev/unet.py:75-87); HS = 32 or 64 (else -20).
// out[B*T][ldo] (C = NH*HS channels); lse[B][NH][T] = log2-domain logsumexp of the scaled scores.
void attn_init();
int attn_fwd(const bf16* qkv, int ld, int B, int T, int NH, int HS, bf16* out, int ldo, float* lse, cudaStream_t st);
// dqkv[B*T][ldd] from dout[B*T][lddo]; dsum[B][NH][T] is scratch.
int attn_bwd(const bf16* qkv, int ld, const bf16* out, int ldo, const bf16* dout, int lddo, const float* lse, int B,
             int T, int NH, int HS, bf16* dqkv, int ldd, float* dsum, cudaStream_t st);

// ---- small fp32 linears, table driven (one launch for all entries)
struct SmallLinear {
    const float* w;   // (OC, C)
    const float* b;   // (OC)
    const float* inp; // (N, C)
    float* out;       // (N, OC)
    int C, OC;
    int silu_in;      // apply SiLU to inp on the fly
    // backward
    const float* dout; // (N, OC)
    float* dw;         // (OC, C)   overwritten
    float* db;         // (OC)      overwritten
    float* db2;        // optional second copy of db (conv1 bias grad == l_emb bias grad), may be null
    float* dinp;       // (N, C)    += gradient w.r.t. the (activated) input, atomically; may be null
};
void small_linear_fwd(const SmallLinear* table_dev, int n_entries, int N, int max_oc, cudaStream_t st,
                      bool rows_ok = false);
void small_linear_bwd(const SmallLinear* table_dev, int n_entries, int N, int max_oc, int max_c, cudaStream_t st);
void silu_f32(const float* x, float* out, size_t n, cudaStream_t st);
// g[i] = dact[i] * silu'(pre[i])
void dsilu_mul(const float* dact, const float* pre, float* g, size_t n, cudaStream_t st);
// timestep embedding (replaces get_timestep_embeddings, train_unet.cu:3258-3313): out[b][j]=cos(t f_j), [half+j]=sin
void time_mlp_fwd(const float* t, int B, int Cm, int Cemb, int max_period, const float* w0, const float* b0,
                  const float* w1, const float* b1, float* sin_emb, float* h0, float* emb, float* semb,
                  cudaStream_t st, const float* label_w = nullptr, const int* labels = nullptr);
// class-conditional model (dev/unet.py:174-175, 301-303): gradient of the label-embedding rows, dw[y[b]] += demb[b]
void label_emb_bwd(const float* demb, const int* labels, int B, int Cemb, float* dw, cudaStream_t st);
// classifier-free guidance (UbConfig.class_dropout): the labels the embedding reads, eff[b] in [0, K], K = null class.
//   CFG_LABELS_TRAIN: K where labels[b] == -1 or the Philox coin (seed, stream id 0xB, counter (b, step)) is below p,
//                     else labels[b]; also copied to eff[B + b] (the last training step's labels)
//   CFG_LABELS_COPY:  labels[b], with -1 mapped to K
//   CFG_LABELS_NULL:  K
enum { CFG_LABELS_TRAIN = 0, CFG_LABELS_COPY = 1, CFG_LABELS_NULL = 2 };
void cfg_labels(const int* labels, int* eff, int B, int K, int mode, float p, uint64_t seed, const int* step_dev,
                cudaStream_t st);
void timestep_embedding(const float* t, int B, int dim, int max_period, float* out, cudaStream_t st);

// ---- diffusion: t ~ U{0..T-1}, eps ~ N(0,1) (Philox4x32-10, counter = element index, key = (seed, step)),
//      x_t = sqrt_ac[t] * x0 + sqrt_1mac[t] * eps.  Replaces sample_timesteps / diffusion_draw_normal /
//      diffusion_forward_by_t (train_unet.cu:3115-3254).  If gen_t / gen_noise are 0 the caller-provided
//      t / noise buffers are used as they are (parity runs inject the oracle's draws).
void diffusion_prepare(const float* x0, const float* sqrt_ac, const float* sqrt_1mac, int B, size_t per_image,
                       int n_timesteps, uint64_t seed, const int* step_dev, int gen_t, int gen_noise, float* t,
                       float* noise, float* x_t, cudaStream_t st, int W = 0, int* flips = nullptr);

// ---- super-resolution conditioning (guided-diffusion SuperResModel): cond (B,C,H,W) fp32 = bilinear upsampling
//      (align_corners = False) of a (B,C,H/f,W/f) image -- full = 0: src is that image (the caller's low-res batch);
//      full = 1: src is the step's x0 (B,C,H,W) and the image is its f x f area means (super_res_train.py's condition),
//      mirrored left-right for the images with flips[b] = 1 (flips may be null)
void superres_cond(const float* src, int full, const int* flips, int B, int C, int H, int W, int f, float* cond,
                   cudaStream_t st);

// ---- weight packing: fp32 master (Cout, Cin, ntaps) -> bf16 fprop pack [tap][Cout][Cin] and (optional) dgrad pack
//      [ntaps-1-tap][Cin][Cout]
struct PackEntry {
    const float* w;
    bf16* wf;  // may be null
    bf16* wd;  // may be null
    int Cout, Cin, ntaps;
};
void pack_weights(const PackEntry* table_dev, int n_entries, int max_tiles, cudaStream_t st);

// ---- AdamW (replaces adamw_kernel2 + unet_zero_grad, train_unet.cu:4706-4757): reads the step counter from
//      device memory, applies grad_scale (1/world for data parallel), and zeroes the gradient.
void adamw_step(float* p, float* g, float* m, float* v, size_t n, float lr, float b1, float b2, float eps, float wd,
                float grad_scale, const int* step_dev, cudaStream_t st, const float* hp_dev = nullptr,
                float* ema = nullptr, float ema_rate = 0.f);  // ema: optional moving average of the parameters
void increment_step(int* step_dev, cudaStream_t st);

// ---- DDPM sampling step (generate.py:29-52).  t_dev holds the current t (2 <= t < T): fill t for the embedding,
//      then (after the forward) x <- mu(x, eps, t) + sigma_t * z and t_dev <- t - 1.
void sample_set_t(const int* t_dev, int B, float* tsteps, cudaStream_t st);
// z: injected noise for this iteration (may be null: Philox(seed, counter = iteration index from it_dev))
void ddpm_step(float* x, const float* eps, const float* betas, const float* sqrt_ac, const float* sqrt_1mac,
               const float* z, size_t n, uint64_t seed, int* t_dev, int* it_dev, cudaStream_t st);
// x ~ N(0,1) (Philox4x32-10, key = seed, stream id 0x2)
void fill_normal(float* x, size_t n, uint64_t seed, cudaStream_t st);

// ---- respaced sampling (guided-diffusion SpacedDiffusion: ddim_sample_loop / p_sample_loop).  Row `it` holds the
//      float32 coefficients of loop iteration it (largest timestep first), built by the host in float64; both samplers
//      share the update
//        x0 = r * x - rm1 * eps  (clamped to [-1, 1] when clip != 0);   x <- c_x0 * x0 + c_x * x + sigma * z
//      (pad: {log beta', lpost'} of a learned-variance model's ancestral rows, else 0)
//      The iteration counter and the Philox key live in device memory, so one captured graph serves every iteration and
//      every seed.
struct SpacedRow {
    float r, rm1, c_x0, c_x, sigma, clip, pad[2];
};
struct SpacedState {
    int it;
    int pad;
    unsigned long long seed;
};
// tsteps[b] = float(ts_table[it]) (the model sees the original timestep)
void spaced_set_t(const int* ts_table, const SpacedState* s, int B, float* tsteps, cudaStream_t st);
// z: injected noise of this iteration (may be null: Philox(seed, stream id 0x5, counter = it)); no draw where sigma = 0.
// Then it <- it + 1.  img3 > 0: learned-variance model -- eps is the (B, 6, H, W) model output [eps | v] with img3 =
// 3 H W floats per image of x, and the row's pad holds {log beta', lpost'} of the learned-range variance (see misc_ops.cu)
// eps_c != null: classifier-free guidance -- eps holds the null-class output, eps_c the conditional one (same layout),
// and the step uses eps_u + s (eps_c - eps_u), s = *scale (device memory); a learned-variance model's v is eps_c's.
void spaced_step(float* x, const float* eps, const SpacedRow* rows, const float* z, size_t n, SpacedState* s,
                 cudaStream_t st, size_t img3 = 0, const float* eps_c = nullptr, const float* scale = nullptr);
// occupy the stream for ~us microseconds (profiling aid: lets the host queue work ahead of the device)
void stream_delay(unsigned us, cudaStream_t st);

}  // namespace ub
