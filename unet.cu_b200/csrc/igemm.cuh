// Parameter blocks + host launch API of the tcgen05 implicit-GEMM kernels (NHWC bf16 operands).
//
//   igemm_conv : fprop AND dgrad of 3x3 (pad 1, stride 1) / 1x1 convolutions and Linear layers
//                D[pix, n] = sum_seg sum_tap sum_c  A_seg[pix + shift(tap), c] * Wp_seg[tap][n][c]
//                replaces conv2d_k3_forward3 / dx_backward (/root/reference/dev/conv2d_k3.cu:679,1132),
//                conv2d_k1_forward2 (dev/conv2d_k1.cu:215) and matmul_forward2 (dev/linear.cu).
//   igemm_wgrad: weight gradient  dW[tap][o][c] = sum_pix dY[pix, o] * X[pix + shift(tap), c]
//                replaces dweight_dbias_backward1 + dweight_reduce_kernel (dev/conv2d_k3.cu:2468,1365).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace ub {

enum OutMode : int {
    OUT_NHWC_BF16 = 0,  // out[((b*H+h)*W+w)*ldo + n]  bf16   (internal layout)
    OUT_NCHW_F32 = 1,   // out[((b*Cout+n)*H+h)*W+w]   fp32   (reference API layout)
    OUT_NHWC_F32 = 2,   // out[((b*H+h)*W+w)*ldo + n]  fp32
};

struct IgemmSeg {
    CUtensorMap tmA;  // activations NHWC bf16, dims (C, W, H, B), box (64, TW, TH, TB), SWIZZLE_128B
    CUtensorMap tmW;  // packed weights [ntaps*Cout][Cin] bf16, dims (Cin, ntaps*Cout), box (64, BN), SWIZZLE_128B
    int cblocks;      // ceil(Cin / 64)
    int ntaps;        // 9 or 1
    const __nv_bfloat16* wp;  // the packed weights behind tmW (L2 prefetch in the prologue)
    int Cin;
};

// The resolved epilogue of both conv kernels (igemm_epi_plan): what epilogue.cuh applies to the accumulator.
struct IgemmEpiParams {
    const float* bias;             // [Cout] or nullptr
    const float* bias2;            // second [Cout] bias (fused 1x1 skip conv) or nullptr
    const float* rowvec;           // [B][Cout] per-image additive vector (time-embedding) or nullptr
    const __nv_bfloat16* residual; // NHWC bf16 [B,H,W,ldr] added to the output, or nullptr
    int ldr;
    void* out;
    int ldo;  // channel pitch of an NHWC output (>= Cout; lets a producer write into a concat buffer)
    int out_mode;
    // fused GroupNorm hooks (see epilogue.cuh); NHWC bf16 output
    float* stats;                   // [B][Cout][2] += (sum, sumsq) of the output, or nullptr
    const __nv_bfloat16* gn_x;      // gn-bwd: GroupNorm input (Cout channels, pitch gn_ldx), or nullptr
    int gn_ldx;
    const float* gn_chsum;          // forward statistics of gn_x [B][Cout][2]
    const float* gn_gamma;
    const float* gn_beta;
    float* gn_S;                    // [B][Cout][2] += (sum dz, sum dz*xhat)
    int gn_silu, gn_cpg;
};

struct IgemmConvParams {
    IgemmSeg seg[2];
    int nseg;
    int B, H, W, Cout;
    int TW, TH, TB;  // pixel tile (TW*TH*TB <= 128)
    int tiles_w, tiles_h, tiles_b;
    int BN;          // output-channel tile: multiple of 16, <= 256
    int stages;
    int tmem_cols;   // power of two >= max(32, nacc * BN)
    int nacc;        // MMA issue streams = accumulators (1, or 2 for grids of at most one CTA per SM); nacc == 2
                     // also has two TMA producer warps (even / odd K blocks)
    int ncomb;       // rows of the staged per-channel addend (TB when a per-image vector is fused, else 1)
    uint32_t a_bytes, b_bytes;  // TMA transaction bytes per stage
    uint32_t stage_bytes;       // smem bytes per stage (A tile 16 KiB + B tile, 1024-aligned)
    IgemmEpiParams epi;         // with a GroupNorm hook: BN % 32 == 0 and a warp's 32 pixels in one image
    int ngimg;                      // rows of the staged GroupNorm constants (TB when gn_x is set, else 0)
    int nred;                       // BN-float rows of the cross-warp reduction scratch (8 with a hook, else 0)
    // GroupNorm statistics on the tensor core (the plain statistics hook on full tiles) --
    // the epilogue stages the bf16 output tile Y in shared memory as an MN-major SW128 operand (the layout TMA gives
    // the wgrad kernel), a ones-tile MMA (the wgrad kernel's bias-gradient trick) leaves sum(y) of channel c in TMEM
    // lane c, the Gram matrix Y^T Y of each image (over the dead accumulator columns) holds the exact sum(y*y) of
    // channel c in lane c, column c, and the Y tile goes to global memory with one TMA store per 64 channels.
    int ms;
    CUtensorMap tmO;                // output tensor, box (64, TW, TH, TB), SWIZZLE_128B (ms only)
};

// persistent row-tile variant (igemm_rows.cu); same segments and epilogue block as IgemmConvParams
struct IgemmRowsParams {
    IgemmSeg seg[2];  // tmA box = (64, W, box_rows, 1), tmW box = (64, BN)
    int nseg;
    int B, H, W, Cout;
    int TH;             // image rows per tile (256 / W)
    int box_rows;       // TH + 2 when a segment is 3x3, else TH
    int tiles_per_img;  // ceil(H / TH)
    int num_tiles;      // B * tiles_per_img * (Cout / BN)
    int BN;             // <= 128
    int a_stages, w_stages;
    int w_resident;     // the weight ring holds the layer's whole weight set (ntaps tiles), loaded once per CTA
    int grid;
    uint32_t a_bytes, a_stage_bytes, w_bytes, w_stage_bytes;
    IgemmEpiParams epi;
};

struct IgemmWgradParams {
    CUtensorMap tmDY;  // dY NHWC bf16 dims (Cout, W, H, B), box (64, TW, TH, TB), TW*TH*TB == 64
    CUtensorMap tmX;   // X  NHWC bf16 dims (Cin,  W, H, B), same box
    int B, H, W, Cin, Cout, ntaps;
    int TW, TH, TB;
    int tiles_w, tiles_h, tiles_b;
    int MO;      // Cout tile: 64 or 128
    int NC;      // Cin tile: multiple of 64, <= 256
    int TC;      // taps per CTA: 3 (one filter row) or 1
    int nsplit;  // split of the pixel (K) dimension across CTAs
    int KP;      // pixels per K tile (= per stage): 64 or 128; an operand atom is KP rows of 128 B
    int stages;
    // column mode (3x3): blockIdx.y = filter column; the three dy taps come from one halo box (64, TW, TH + 2, TB) per
    // 64-channel atom of X (tmX then has that box), hatom bytes each; accumulator columns [atom][dy][64]
    int colmode;
    uint32_t hatom;
    int lg_img;  // log2(TW * TH): pixels of one image inside a K tile
    int tmem_cols;
    uint32_t stage_bytes, tx_bytes;
    float* partial;  // [nsplit][ntaps][Cout][Cin] fp32 (two-pass mode: igemm_wgrad_reduce sums the splits)
    // accumulate mode (trainer): every CTA adds its tile into acc[ntaps][Cout][Cin] (TMA reduce-add, see tmAcc) -- no
    // partial buffer, no per-layer reduce launch; wgrad_finalize turns [tap][o][c] into the reference [o][c][tap]
    // layout for a whole gradient bucket at once (for 1x1 / linear layers acc IS the final gradient).
    float* acc;
    // accumulate mode: the epilogue stages its accumulator rows in the (idle) operand ring and adds them with TMA
    // reduce-add boxes of 32 columns x MO/4 rows (one epilogue warp's rows) instead of per-lane REDs, whose
    // thread-per-row addresses cost one LSU pass per lane.  tmAcc: fp32, dims (Cin, ntaps*Cout), 128B swizzle.
    CUtensorMap tmAcc;
    // fused bias gradient: the CTAs of the centre tap / first Cin tile also contract dY with a tile of ones
    // (one extra N=16 MMA per K step), and add column 0 of that accumulator into dbias (and dbias2) atomically.
    float* dbias;
    float* dbias2;
    uint32_t ones_off;  // byte offset of the 8 KiB ones tile behind the stages (0 = no bias fusion)
};
struct WgradFinalizeEntry {
    float* acc;  // [9][Cout][Cin], zeroed again by the finalize kernel
    float* dw;   // [Cout][Cin][9]
    int Cout, Cin;
};

// ---- host API (implemented in igemm.cu); all return cudaError_t-like int (0 == ok) -------------------------
struct ConvSegDesc {
    const __nv_bfloat16* x;  // NHWC bf16 [B,H,W,ldx]; channels [0,Cin) are used
    int Cin;
    int ldx;                   // channel pitch of x
    const __nv_bfloat16* wp;   // packed [ntaps][Cout][Cin] bf16
    int ntaps;
};
struct ConvEpilogue {
    const float* bias = nullptr;
    const float* bias2 = nullptr;
    const float* rowvec = nullptr;
    const __nv_bfloat16* residual = nullptr;
    int ldr = 0;
    void* out = nullptr;
    int ldo = 0;
    int out_mode = OUT_NHWC_BF16;
    // fused GroupNorm hooks
    float* stats = nullptr;
    const __nv_bfloat16* gn_x = nullptr;
    int gn_ldx = 0;
    const float* gn_chsum = nullptr;
    const float* gn_gamma = nullptr;
    const float* gn_beta = nullptr;
    float* gn_S = nullptr;
    int gn_silu = 0, gn_groups = 32;
};
// Fills `e` from `ep` (ldr, ldo default to Cout; gn_cpg = Cout / gn_groups) and checks the epilogue contract both conv
// kernels share.  Returns 0 or -15 (GroupNorm hook), -6 (output), -7 (residual), -8 (bias, bias2, rowvec).  The
// planners add the checks that depend on their tiling.
int igemm_epi_plan(IgemmEpiParams* e, const ConvEpilogue& ep, int Cout);
// TMA maps (bf16, 128-byte swizzle, zero fill out of bounds).  make_act_map: NHWC activations, dims (C, W, H, B),
// channel pitch ld, box (64, TW, TH, TB); -11 misaligned, -12 encode failed.  make_bf16_map_2d: row-major
// [rows][cols] with pitch ld, box (64, box_rows); -13 misaligned, -14 encode failed.  Both: -10 no driver entry point.
int make_act_map(CUtensorMap* m, const __nv_bfloat16* x, int C, int ld, int W, int H, int B, int TW, int TH, int TB);
int make_bf16_map_2d(CUtensorMap* m, const __nv_bfloat16* base, int cols, int rows, int ld, int box_rows);
// One-time kernel attribute setup (opt-in shared memory); safe to call repeatedly, call before graph capture.
void igemm_init();
// Fills `p` (tensor maps + tiling). Returns 0 or a negative error code (unsupported shape).
int igemm_conv_plan(IgemmConvParams* p, const ConvSegDesc* segs, int nseg, int B, int H, int W, int Cout,
                    const ConvEpilogue& ep);
int igemm_conv_launch(const IgemmConvParams& p, cudaStream_t st);

bool igemm_rows_eligible(int B, int H, int W, int Cout);
int igemm_rows_plan(IgemmRowsParams* p, const ConvSegDesc* segs, int nseg, int B, int H, int W, int Cout,
                    const ConvEpilogue& ep, int sm_count);
int igemm_rows_launch(const IgemmRowsParams& p, cudaStream_t st);
void igemm_rows_init();

int igemm_wgrad_plan(IgemmWgradParams* p, const __nv_bfloat16* dy, int ldy, const __nv_bfloat16* x, int ldx, int B,
                     int H, int W, int Cin, int Cout, int ntaps, float* partial, size_t partial_cap_floats,
                     int sm_count);
// accumulate mode: acc [ntaps][Cout][Cin] must hold zeros (or the running sum); dbias/dbias2 may be null
int igemm_wgrad_plan_acc(IgemmWgradParams* p, const __nv_bfloat16* dy, int ldy, const __nv_bfloat16* x, int ldx, int B,
                         int H, int W, int Cin, int Cout, int ntaps, float* acc, float* dbias, float* dbias2,
                         int sm_count);
// dw[o][c][tap] = acc[tap][o][c]; acc = 0, for n entries of a device table (max_elems = max Cout*Cin over them)
int igemm_wgrad_finalize(const WgradFinalizeEntry* table_dev, int n_entries, size_t max_elems, cudaStream_t st);
int igemm_wgrad_launch(const IgemmWgradParams& p, cudaStream_t st);
// dW (reference layout [Cout][Cin][ntaps], fp32) = sum over splits of partial[split][tap][o][c]; overwrite.
int igemm_wgrad_reduce(const IgemmWgradParams& p, float* dweight, cudaStream_t st);
size_t igemm_wgrad_partial_floats(int Cin, int Cout, int ntaps, int nsplit);

#ifdef UB_TRACE
void igemm_trace_dump(int nctas, double clock_ghz);  // phase timeline of the last igemm_conv_kernel launch
void igemm_trace_set_mode(int m);                    // 0 normal, 1 TMA stream only, 2 MMA stream only
void igemm_rows_trace_dump(int nctas, int ntiles_total);  // per-tile phase timeline of the last igemm_rows_kernel launch
#endif

}  // namespace ub
