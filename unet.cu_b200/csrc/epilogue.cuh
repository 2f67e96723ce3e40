// Shared epilogue of the implicit-GEMM kernels: one thread owns one output pixel (TMEM lane) and NC consecutive
// output channels.  The per-channel addend (bias + second bias + per-image embedding vector) is staged in shared
// memory by the caller BEFORE the accumulator is ready, and the residual row is fetched before the TMEM wait, so
// the only exposed latency per chunk is one tcgen05.wait::ld (the first version waited on dependent global loads per
// 16-column chunk, which made the epilogue -- not the MMA -- the critical path of small-K layers).
//
// Two fused GroupNorm hooks (they remove one full pass over the tensor each, and ~100 launches per step):
//   * stats   : the epilogue of the conv that PRODUCES a tensor accumulates its per-(image, channel) sum and sum of
//               squares, which is all GroupNorm's statistics pass needs (replaces gn_stats).
//   * gn-bwd  : the epilogue of the dgrad conv that produces dL/d(silu(gn(x))) multiplies by silu'(gn(x)) on the
//               spot, writes dz = dL/d(gn(x)) instead, and accumulates the per-(image, channel) sums of dz and
//               dz * xhat (replaces gn_bwd_stats; gn_bwd_apply then needs no sigmoid at all).
// Both reduce over the 32 pixels of a warp by a 31-shuffle transpose-reduce and add the warp totals of the CTA's
// epilogue warps in shared memory; one red.global.add.v2.f32 per (tile, channel) follows.
#pragma once
#include "igemm.cuh"
#include "ptx.cuh"

namespace ub {

struct EpiOut {
    const __nv_bfloat16* residual;
    int ldr;
    void* out;
    int ldo;
    int out_mode;
    int Cout, H, W;
    // fused GroupNorm hooks (NHWC bf16 output only)
    float* stats = nullptr;              // [B][Cout][2] += (sum, sumsq) of the stored (bf16-rounded) output
    const __nv_bfloat16* gx = nullptr;   // gn-bwd: the GroupNorm input x, NHWC bf16 [.., ldgx]
    int ldgx = 0;
    float* gS = nullptr;                 // gn-bwd: [B][Cout][2] += (sum dz, sum dz*xhat)
    int gsilu = 0;
    // two MMA streams (igemm_conv2_kernel): the result is the sum of two accumulators acc_stride TMEM columns apart
    int nacc = 1;
    uint32_t acc_stride = 0;
};

// the kernel-side view of a conv kernel's epilogue block (one accumulator; the two-stream kernel sets nacc, acc_stride)
__device__ __forceinline__ EpiOut epi_out(const IgemmEpiParams& ep, int Cout, int H, int W) {
    EpiOut e{ep.residual, ep.ldr, ep.out, ep.ldo, ep.out_mode, Cout, H, W};
    e.stats = ep.stats, e.gx = ep.gn_x, e.ldgx = ep.gn_ldx, e.gS = ep.gn_S, e.gsilu = ep.gn_silu;
    return e;
}

// v[0..16) = the 16 accumulator columns at taddr, summed over the kernel's accumulators
__device__ __forceinline__ void epi_tmem_load16(const EpiOut& e, uint32_t taddr, uint32_t (&v)[16]) {
    tmem_ld16(taddr, v);
    if (e.nacc == 2) {
        uint32_t u[16];
        tmem_ld16(taddr + e.acc_stride, u);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
    }
}

__device__ __forceinline__ float epi_sigmoid(float z) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * z));
    return fmaf(0.5f, t, 0.5f);
}

__device__ __forceinline__ void unpack_bf16x8(const uint4& v, float* f) {
    const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h2 = *reinterpret_cast<const __nv_bfloat162*>(&u[i]);
        f[2 * i] = __bfloat162float(h2.x);
        f[2 * i + 1] = __bfloat162float(h2.y);
    }
}

// NC = 16 or 32 columns starting at absolute channel n, TMEM address taddr; comb points at the staged addend of
// channel n (shared memory).
template <int NC>
__device__ __forceinline__ void epi_chunk(const EpiOut& e, uint32_t taddr, const float* comb, bool valid, size_t pix,
                                          int b, int h, int w, int n) {
    uint32_t v[NC];
    if constexpr (NC == 32) {
        tmem_ld32(taddr, v);  // (one accumulator only: epi_row)
    } else {
        epi_tmem_load16(e, taddr, v);
    }
    uint4 r[NC / 8];
    if (e.residual && valid) {
        const uint4* rp = reinterpret_cast<const uint4*>(e.residual + pix * e.ldr + n);
#pragma unroll
        for (int j = 0; j < NC / 8; ++j) r[j] = rp[j];
    }
    tmem_ld_wait();
    if (!valid) return;
    float f[NC];
    const uint32_t comb_s = smem_u32(comb);
#pragma unroll
    for (int j = 0; j < NC; j += 4) {
        const float4 c = lds_v4(comb_s + 4u * j);
        f[j] = __uint_as_float(v[j]) + c.x, f[j + 1] = __uint_as_float(v[j + 1]) + c.y;
        f[j + 2] = __uint_as_float(v[j + 2]) + c.z, f[j + 3] = __uint_as_float(v[j + 3]) + c.w;
    }
    if (e.residual) {
#pragma unroll
        for (int j = 0; j < NC / 8; ++j) {
            float t[8];
            unpack_bf16x8(r[j], t);
#pragma unroll
            for (int i = 0; i < 8; ++i) f[j * 8 + i] += t[i];
        }
    }
    if (e.out_mode == OUT_NHWC_BF16) {
        __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(e.out) + pix * e.ldo + n;
#pragma unroll
        for (int j = 0; j < NC / 8; ++j) {
            uint32_t pk[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const __nv_bfloat162 h2 = __floats2bfloat162_rn(f[j * 8 + 2 * i], f[j * 8 + 2 * i + 1]);
                pk[i] = *reinterpret_cast<const uint32_t*>(&h2);
            }
            reinterpret_cast<uint4*>(op)[j] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
    } else if (e.out_mode == OUT_NHWC_F32) {
        float* op = reinterpret_cast<float*>(e.out) + pix * e.ldo + n;
#pragma unroll
        for (int j = 0; j < NC; j += 4)
            *reinterpret_cast<float4*>(op + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
    } else {  // OUT_NCHW_F32: a warp writes 32 consecutive pixels of one channel -> coalesced
        float* op = reinterpret_cast<float*>(e.out) + ((size_t(b) * e.Cout + n) * e.H + h) * e.W + w;
        const size_t cs = size_t(e.H) * e.W;
#pragma unroll
        for (int j = 0; j < NC; ++j) op[j * cs] = f[j];
    }
}

// 16-column chunk with one of the GroupNorm hooks (NHWC bf16 output).  Every lane of the warp takes part in the
// reduction; lanes whose pixel is outside the tensor contribute zeros and store nothing.  All pixels of a warp belong
// to one image (the plan guarantees it).  gconst = staged [4][BN] per-channel constants of that image (a = gamma*rstd,
// bb = beta - mean*a, rstd, mean*rstd), offset to this chunk's first column (gn-bwd only); cstride = BN.
// xr holds the 16 channels [n, n+16) of the pixel's side input -- the residual row (stats mode) or the GroupNorm input
// row (gn-bwd mode), never both (plan) -- fetched one chunk AHEAD (epi_side_load): a dependent global load per chunk
// was the longest stall of the hooked epilogue.  On return xr holds the chunk at channel n_next (if n_next >= 0).
__device__ __forceinline__ void epi_side_load(const EpiOut& e, bool valid, size_t pix, int n, uint4 (&xr)[2]) {
    if ((e.residual || e.gx) && valid) {
        const uint4* xp = e.gx ? reinterpret_cast<const uint4*>(e.gx + pix * e.ldgx + n)
                               : reinterpret_cast<const uint4*>(e.residual + pix * e.ldr + n);
        xr[0] = xp[0], xr[1] = xp[1];
    }
}
__device__ __forceinline__ void epi_chunk_gn(const EpiOut& e, uint32_t taddr, const float* comb, const float* gconst,
                                             int cstride, bool valid, size_t pix, int n, int lane, float* red,
                                             uint4 (&xr)[2], int n_next) {
    uint32_t v[16];
    epi_tmem_load16(e, taddr, v);
    uint4 xn[2];
    if (n_next >= 0) epi_side_load(e, valid, pix, n_next, xn);
    tmem_ld_wait();
    float f[16], q[16];
    const uint32_t comb_s = smem_u32(comb);
#pragma unroll
    for (int j = 0; j < 16; j += 4) {
        const float4 c = lds_v4(comb_s + 4u * j);
        f[j] = __uint_as_float(v[j]) + c.x, f[j + 1] = __uint_as_float(v[j + 1]) + c.y;
        f[j + 2] = __uint_as_float(v[j + 2]) + c.z, f[j + 3] = __uint_as_float(v[j + 3]) + c.w;
    }
    if (valid) {
        if (e.gx) {
            // f = dL/d(act(gn(x)))  ->  dz = f * act'(z);  q = dz * xhat
            const uint32_t gc_s = smem_u32(gconst), gstride = 4u * uint32_t(cstride);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                float x[8];
                unpack_bf16x8(xr[j], x);
#pragma unroll
                for (int h4 = 0; h4 < 2; ++h4) {  // four channels at a time: one 16-byte read per constant row
                    const uint32_t ga = gc_s + 4u * uint32_t(j * 8 + h4 * 4);
                    const float4 ca = lds_v4(ga), cb = lds_v4(ga + gstride);
                    const float4 cr = lds_v4(ga + 2u * gstride), cm = lds_v4(ga + 3u * gstride);
                    const float a4[4] = {ca.x, ca.y, ca.z, ca.w}, b4[4] = {cb.x, cb.y, cb.z, cb.w};
                    const float r4[4] = {cr.x, cr.y, cr.z, cr.w}, m4[4] = {cm.x, cm.y, cm.z, cm.w};
#pragma unroll
                    for (int i4 = 0; i4 < 4; ++i4) {
                        const int i = h4 * 4 + i4, c = j * 8 + i;
                        float dz = f[c];
                        if (e.gsilu) {
                            const float z = fmaf(x[i], a4[i4], b4[i4]);
                            const float sg = epi_sigmoid(z);
                            dz *= sg * fmaf(z, 1.f - sg, 1.f);
                        }
                        // the stored (bf16) dz is what gn_bwd_apply will read: sum exactly that
                        dz = __bfloat162float(__float2bfloat16(dz));
                        f[c] = dz;
                        q[c] = dz * fmaf(x[i], r4[i4], -m4[i4]);
                    }
                }
            }
        } else {
            if (e.residual) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    float t[8];
                    unpack_bf16x8(xr[j], t);
#pragma unroll
                    for (int i = 0; i < 8; ++i) f[j * 8 + i] += t[i];
                }
            }
            // round to the stored precision first: the statistics then describe exactly the tensor the consumer reads
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                f[c] = __bfloat162float(__float2bfloat16(f[c]));
                q[c] = f[c] * f[c];
            }
        }
        uint32_t pk[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
            pk[i] = *reinterpret_cast<const uint32_t*>(&h2);
        }
        __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(e.out) + pix * e.ldo + n;
        reinterpret_cast<uint4*>(op)[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        reinterpret_cast<uint4*>(op)[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) f[j] = 0.f, q[j] = 0.f;
    }
    // Column sums over the warp's 32 pixels by a transpose-reduce butterfly: 31 shuffles move half as many bytes
    // through the SM's shuffle/shared-memory crossbar as the 8 STS.128 + 32 LDS of the shared-memory transpose
    // (64 wavefronts per chunk and warp; with 16 epilogue warps per SM that pipe is what bounds the hooked epilogue).
    float cs[32];
#pragma unroll
    for (int j = 0; j < 16; ++j) cs[j] = f[j], cs[16 + j] = q[j];
#pragma unroll
    for (int sft = 16; sft >= 1; sft >>= 1) {
        const bool up = (lane & sft) != 0;
#pragma unroll
        for (int i = 0; i < sft; ++i) {
            const float keep = up ? cs[i + sft] : cs[i];
            const float send = up ? cs[i] : cs[i + sft];
            cs[i] = keep + __shfl_xor_sync(0xffffffffu, send, sft);
        }
    }
    // lane L holds the warp's total of cs[L]: f column L for L < 16, q column L - 16 above
    sts_f32(smem_u32(red) + 4u * uint32_t(2 * (lane & 15) + (lane >> 4)), cs[0]);
    xr[0] = xn[0], xr[1] = xn[1];
}

// red[4 quadrants][BN][2] -> global [B][Cout][2].  Called by the nthreads epilogue threads after a barrier; quadrant
// q's 32 pixels belong to tile-local image min(32 q / rows_per_img, TB - 1).
__device__ __forceinline__ void epi_flush_stats(const float* red, float* dst, int Cout, int n0, int BN, int b0,
                                                int B, int rows_per_img, int TB, int tid, int nthreads) {
    for (int c = tid; c < BN; c += nthreads) {
        for (int img = 0; img < TB; ++img) {
            float s = 0.f, ss = 0.f;
            bool any = false;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int iq = min((q * 32) / rows_per_img, TB - 1);
                if (iq == img) {
                    const float2 v = *reinterpret_cast<const float2*>(red + (size_t(q) * BN + c) * 2);
                    s += v.x, ss += v.y, any = true;
                }
            }
            if (any && b0 + img < B) {
                float* d = dst + (size_t(b0 + img) * Cout + n0 + c) * 2;
                asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(d), "f"(s), "f"(ss) : "memory");
            }
        }
    }
}

// Columns [0, BN) of one accumulator row.  The row is shared by `nhalf` warps of the same TMEM lane quadrant: chunk i
// goes to warp i % nhalf.
__device__ __forceinline__ void epi_row(const EpiOut& e, uint32_t trow, const float* comb, int BN, bool valid,
                                        size_t pix, int b, int h, int w, int n0, const float* gconst = nullptr,
                                        int lane = 0, float* red = nullptr, int half = 0, int nhalf = 1,
                                        uint4* side = nullptr) {
    if (e.stats || e.gx) {  // BN % 32 == 0 (plan); red = this quadrant's [BN][2] row of the reduction scratch
        // side = the first chunk's side input, loaded by the caller (epi_side_load at channel n0 + 16 * half) before
        // it waited for the accumulator
        uint4 xr[2] = {side[0], side[1]};
        for (int c0 = 16 * half; c0 < BN; c0 += 16 * nhalf) {
            const int cn = c0 + 16 * nhalf;
            epi_chunk_gn(e, trow + uint32_t(c0), comb + c0, gconst + c0, BN, valid, pix, n0 + c0, lane, red + 2 * c0,
                         xr, cn < BN ? n0 + cn : -1);
        }
        return;
    }
    int i = 0, c0 = 0;
    if (e.nacc == 1)  // (two accumulators are added per 16-column chunk)
        for (; c0 + 32 <= BN; c0 += 32, ++i)
            if (i % nhalf == half) epi_chunk<32>(e, trow + uint32_t(c0), comb + c0, valid, pix, b, h, w, n0 + c0);
    for (; c0 < BN; c0 += 16, ++i)
        if (i % nhalf == half) epi_chunk<16>(e, trow + uint32_t(c0), comb + c0, valid, pix, b, h, w, n0 + c0);
}

// comb[c] = bias[n0+c] + bias2[n0+c] + rowvec[b][n0+c] for c in [0, BN), computed by the calling threads (tid in
// [0, nthreads))
__device__ __forceinline__ void epi_stage_comb(float* comb, const float* bias, const float* bias2, const float* rowvec,
                                               int b, int Cout, int n0, int BN, int tid, int nthreads) {
    for (int c = tid; c < BN; c += nthreads) {
        float v = 0.f;
        if (bias) v += bias[n0 + c];
        if (bias2) v += bias2[n0 + c];
        if (rowvec) v += rowvec[size_t(b) * Cout + n0 + c];
        comb[c] = v;
    }
}

// gconst[0..3][BN] for image b, channels [n0, n0+BN): a = gamma*rstd, bb = beta - mean*a, rstd, mean*rstd, from the
// forward statistics chsum[B][C][2] (per-channel sum / sumsq over the HW pixels), groups of cpg channels.
__device__ __forceinline__ void epi_stage_gconst(float* gconst, const float* chsum, const float* gamma,
                                                 const float* beta, int b, int C, int cpg, int HW, int n0, int BN,
                                                 int tid, int nthreads) {
    for (int c = tid; c < BN; c += nthreads) {
        const int ch = n0 + c;
        const int g0 = (ch / cpg) * cpg;
        const float* cs = chsum + (size_t(b) * C + g0) * 2;
        float s = 0.f, ss = 0.f;
        for (int k = 0; k < cpg; ++k) s += cs[2 * k], ss += cs[2 * k + 1];
        const float n = float(cpg) * float(HW);
        const float mean = s / n;
        const float var = fmaxf(ss / n - mean * mean, 0.f);
        const float r = rsqrtf(var + 1e-5f);
        const float a = r * gamma[ch];
        gconst[c] = a;
        gconst[BN + c] = beta[ch] - mean * a;
        gconst[2 * BN + c] = r;
        gconst[3 * BN + c] = mean * r;
    }
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace ub
