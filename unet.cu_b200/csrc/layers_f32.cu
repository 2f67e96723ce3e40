// See layers_f32.cuh.
#include "layers_f32.cuh"
#include "launch.cuh"

namespace ub {
namespace f32 {

static inline unsigned grid_for(size_t n, int threads, int waves = 8) {
    size_t b = (n + threads - 1) / threads;
    const size_t cap = size_t(sm_count()) * waves;  // (launch.cuh: 148 on a B200)
    return unsigned(b < cap ? (b ? b : 1) : cap);
}

__device__ __forceinline__ float block_sum(float v, float* red) {
    for (int off = 16; off; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    if (threadIdx.x < 32) {
        for (int off = 16; off; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (threadIdx.x == 0) red[0] = t;
    }
    __syncthreads();
    return red[0];
}

// ------------------------------------------------------------------------------------------------ layout
__global__ void nchw_to_nhwc_bf16_kernel(const float* __restrict__ x, int C, int HW, __nv_bfloat16* __restrict__ y) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, p = p0 + tx;
        tile[i][tx] = (c < C && p < HW) ? x[(size_t(b) * C + c) * HW + p] : 0.f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int p = p0 + i, c = c0 + tx;
        if (p < HW && c < C) y[(size_t(b) * HW + p) * C + c] = __float2bfloat16(tile[tx][i]);
    }
}
// The same conversion for HW % 4 == 0, C % 2 == 0 (every tensor-core shape): a block moves a 64-channel x 64-pixel tile.
// Read side: every thread has four 16-byte loads in flight (two channels x 4 pixels, twice), 16 lanes cover 256
// contiguous bytes of a channel row.  The pair (c, c+1) is rounded to bf16 and parked as one 32-bit word in a
// [pixel][channel-pair] tile with an odd pitch (33 words: 2-way conflicts on the stores, none on the reads).  Write side:
// a warp owns a pixel and stores its 64 channels as one 128-byte row -- the row the TMA boxes of the conv kernels read.
// (The 32 x 32 kernel above moved 4 KiB per block with one 4-byte load per thread in flight and wrote 64-byte half rows:
// 1.8 TB/s on a 100 MB tensor; this one is sized for the HBM roofline of 6 B per element.)
__global__ void __launch_bounds__(256) nchw_to_nhwc_bf16_tile64_kernel(const float* __restrict__ x, int C, int HW,
                                                                       __nv_bfloat16* __restrict__ y) {
    __shared__ uint32_t tile[64][33];  // [pixel][channel pair]
    const int b = blockIdx.z, p0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
    float4 v[2][2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int idx = threadIdx.x + 256 * k;  // 32 channel pairs x 16 pixel quads
        const int cp = idx >> 4, q = idx & 15;
        const int c = c0 + 2 * cp, p = p0 + 4 * q;
        const bool ok = c < C && p < HW;        // (C even, HW % 4 == 0: a pair / quad is inside or outside as a whole)
        const float* src = x + (size_t(b) * C + c) * HW + p;
        v[k][0] = ok ? __ldg(reinterpret_cast<const float4*>(src)) : make_float4(0.f, 0.f, 0.f, 0.f);
        v[k][1] = ok ? __ldg(reinterpret_cast<const float4*>(src + HW)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int idx = threadIdx.x + 256 * k;
        const int cp = idx >> 4, q = idx & 15;
        const float a[4] = {v[k][0].x, v[k][0].y, v[k][0].z, v[k][0].w};
        const float d[4] = {v[k][1].x, v[k][1].y, v[k][1].z, v[k][1].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(a[j], d[j]);
            tile[4 * q + j][cp] = *reinterpret_cast<const uint32_t*>(&h2);
        }
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (c0 + 2 * lane < C) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int pl = warp + 8 * i;
            if (p0 + pl < HW)
                *reinterpret_cast<uint32_t*>(y + (size_t(b) * HW + p0 + pl) * C + c0 + 2 * lane) = tile[pl][lane];
        }
    }
}
void nchw_to_nhwc_bf16(const float* x, int B, int C, int HW, __nv_bfloat16* y, cudaStream_t st) {
    if (HW % 4 == 0 && C % 2 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
        (reinterpret_cast<uintptr_t>(y) & 3) == 0) {
        dim3 grid((HW + 63) / 64, (C + 63) / 64, B);
        nchw_to_nhwc_bf16_tile64_kernel<<<grid, 256, 0, st>>>(x, C, HW, y);
        return;
    }
    dim3 grid((HW + 31) / 32, (C + 31) / 32, B);
    nchw_to_nhwc_bf16_kernel<<<grid, dim3(32, 8), 0, st>>>(x, C, HW, y);
}
__global__ void cast_bf16_kernel(const float* __restrict__ x, size_t n, __nv_bfloat16* __restrict__ y) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x)
        y[i] = __float2bfloat16(x[i]);
}
void cast_bf16(const float* x, size_t n, __nv_bfloat16* y, cudaStream_t st) {
    cast_bf16_kernel<<<grid_for(n, 256), 256, 0, st>>>(x, n, y);
}

// ------------------------------------------------------------------------------------------------ GroupNorm
__global__ void groupnorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                     const float* __restrict__ b, float* __restrict__ out, float* __restrict__ mean,
                                     float* __restrict__ rstd, int C, int HW, int G) {
    __shared__ float red[32];
    const int bg = blockIdx.x;  // b * G + g
    const int g = bg % G, cpg = C / G;
    const size_t n = size_t(cpg) * HW;
    const float* xp = x + size_t(bg) * n;  // groups are contiguous in NCHW
    float* op = out + size_t(bg) * n;
    float s = 0.f;
    for (size_t i = threadIdx.x; i < n; i += blockDim.x) s += xp[i];
    const float m = block_sum(s, red) / float(n);
    float v = 0.f;
    for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
        const float d = xp[i] - m;
        v += d * d;
    }
    const float r = rsqrtf(block_sum(v, red) / float(n) + 1e-5f);
    if (threadIdx.x == 0) {
        if (mean) mean[bg] = m;
        if (rstd) rstd[bg] = r;
    }
    for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
        const int c = g * cpg + int(i / HW);
        op[i] = (xp[i] - m) * r * w[c] + b[c];
    }
}
void groupnorm_fwd(const float* x, const float* w, const float* b, float* out, float* mean, float* rstd, int B, int C,
                   int HW, int G, cudaStream_t st) {
    groupnorm_fwd_kernel<<<B * G, 512, 0, st>>>(x, w, b, out, mean, rstd, C, HW, G);
}

__global__ void groupnorm_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ x,
                                     const float* __restrict__ mean, const float* __restrict__ rstd,
                                     const float* __restrict__ w, float* __restrict__ dx, float* __restrict__ dw,
                                     float* __restrict__ db, int C, int HW, int G) {
    __shared__ float red[32];
    const int bg = blockIdx.x;
    const int g = bg % G, cpg = C / G;
    const size_t n = size_t(cpg) * HW;
    const float* xp = x + size_t(bg) * n;
    const float* dp = dout + size_t(bg) * n;
    float* op = dx + size_t(bg) * n;
    const float m = mean[bg], r = rstd[bg];
    float g1 = 0.f, g2 = 0.f;
    for (int cc = 0; cc < cpg; ++cc) {
        const int c = g * cpg + cc;
        float s1 = 0.f, s2 = 0.f;
        for (int i = threadIdx.x; i < HW; i += blockDim.x) {
            const float d = dp[size_t(cc) * HW + i];
            s1 += d;
            s2 += d * (xp[size_t(cc) * HW + i] - m) * r;
        }
        s1 = block_sum(s1, red);
        s2 = block_sum(s2, red);
        if (threadIdx.x == 0) {
            atomicAdd(&db[c], s1);
            atomicAdd(&dw[c], s2);
        }
        g1 += w[c] * s1;
        g2 += w[c] * s2;
    }
    g1 /= float(n), g2 /= float(n);
    for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
        const int c = g * cpg + int(i / HW);
        const float xh = (xp[i] - m) * r;
        op[i] = r * (dp[i] * w[c] - g1 - xh * g2);
    }
}
void groupnorm_bwd(const float* dout, const float* x, const float* mean, const float* rstd, const float* w, float* dx,
                   float* dw, float* db, int B, int C, int HW, int G, cudaStream_t st) {
    groupnorm_bwd_kernel<<<B * G, 512, 0, st>>>(dout, x, mean, rstd, w, dx, dw, db, C, HW, G);
}

// ------------------------------------------------------------------------------------------------ elementwise
__global__ void silu_fwd_kernel(const float* __restrict__ x, float* __restrict__ out, size_t n) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        const float v = x[i];
        out[i] = v / (1.f + expf(-v));
    }
}
__global__ void silu_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ x, float* __restrict__ dx,
                                size_t n) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        const float v = x[i];
        const float s = 1.f / (1.f + expf(-v));
        dx[i] = dout[i] * s * (1.f + v * (1.f - s));
    }
}
__global__ void add_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out,
                           size_t n) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x)
        out[i] = a[i] + b[i];
}
void silu_fwd(const float* x, float* out, size_t n, cudaStream_t st) {
    silu_fwd_kernel<<<grid_for(n, 256), 256, 0, st>>>(x, out, n);
}
void silu_bwd(const float* dout, const float* x, float* dx, size_t n, cudaStream_t st) {
    silu_bwd_kernel<<<grid_for(n, 256), 256, 0, st>>>(dout, x, dx, n);
}
void add(const float* a, const float* b, float* out, size_t n, cudaStream_t st) {
    add_kernel<<<grid_for(n, 256), 256, 0, st>>>(a, b, out, n);
}

// ------------------------------------------------------------------------------------------------ resampling
__global__ void upsample_fwd_kernel(float* __restrict__ out, const float* __restrict__ x, size_t total, int H, int W) {
    const int Wo = 2 * W, Ho = 2 * H;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int wo = int(i % Wo), ho = int((i / Wo) % Ho);
        const size_t bc = i / (size_t(Wo) * Ho);
        out[i] = x[(bc * H + ho / 2) * W + wo / 2];
    }
}
__global__ void upsample_bwd_kernel(float* __restrict__ dx, const float* __restrict__ dout, size_t total, int H,
                                    int W) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int w = int(i % W), h = int((i / W) % H);
        const size_t bc = i / (size_t(W) * H);
        const float* p = dout + (bc * 2 * H + 2 * h) * (2 * W) + 2 * w;
        dx[i] = p[0] + p[1] + p[2 * W] + p[2 * W + 1];
    }
}
__global__ void avgpool_fwd_kernel(float* __restrict__ out, const float* __restrict__ x, size_t total, int H, int W) {
    const int Wo = W / 2, Ho = H / 2;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int wo = int(i % Wo), ho = int((i / Wo) % Ho);
        const size_t bc = i / (size_t(Wo) * Ho);
        const float* p = x + (bc * H + 2 * ho) * W + 2 * wo;
        out[i] = 0.25f * (p[0] + p[1] + p[W] + p[W + 1]);
    }
}
__global__ void avgpool_bwd_kernel(const float* __restrict__ dout, float* __restrict__ dx, size_t total, int H,
                                   int W) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int w = int(i % W), h = int((i / W) % H);
        const size_t bc = i / (size_t(W) * H);
        dx[i] = 0.25f * dout[(bc * (H / 2) + h / 2) * (W / 2) + w / 2];
    }
}
void upsample_fwd(float* out, const float* x, size_t BC, int H, int W, cudaStream_t st) {
    const size_t total = BC * 4 * H * W;
    upsample_fwd_kernel<<<grid_for(total, 256), 256, 0, st>>>(out, x, total, H, W);
}
void upsample_bwd(float* dx, const float* dout, size_t BC, int H, int W, cudaStream_t st) {
    const size_t total = BC * H * W;
    upsample_bwd_kernel<<<grid_for(total, 256), 256, 0, st>>>(dx, dout, total, H, W);
}
void avgpool_fwd(float* out, const float* x, size_t BC, int H, int W, cudaStream_t st) {
    const size_t total = BC * (H / 2) * (W / 2);
    avgpool_fwd_kernel<<<grid_for(total, 256), 256, 0, st>>>(out, x, total, H, W);
}
void avgpool_bwd(const float* dout, float* dx, size_t BC, int H, int W, cudaStream_t st) {
    const size_t total = BC * H * W;
    avgpool_bwd_kernel<<<grid_for(total, 256), 256, 0, st>>>(dout, dx, total, H, W);
}

// ------------------------------------------------------------------------------------------------ concat / broadcast
__global__ void concat_fwd_kernel(const float* __restrict__ x1, const float* __restrict__ x2, float* __restrict__ out,
                                  size_t total, size_t n1, size_t n2) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const size_t b = i / (n1 + n2), r = i % (n1 + n2);
        out[i] = r < n1 ? x1[b * n1 + r] : x2[b * n2 + (r - n1)];
    }
}
__global__ void concat_bwd_kernel(const float* __restrict__ dout, float* __restrict__ dx1, float* __restrict__ dx2,
                                  size_t total, size_t n1, size_t n2) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const size_t b = i / (n1 + n2), r = i % (n1 + n2);
        if (r < n1)
            dx1[b * n1 + r] = dout[i];
        else
            dx2[b * n2 + (r - n1)] = dout[i];
    }
}
void concat_fwd(const float* x1, const float* x2, float* out, int B, int C1, int C2, int HW, cudaStream_t st) {
    const size_t n1 = size_t(C1) * HW, n2 = size_t(C2) * HW, total = size_t(B) * (n1 + n2);
    concat_fwd_kernel<<<grid_for(total, 256), 256, 0, st>>>(x1, x2, out, total, n1, n2);
}
void concat_bwd(const float* dout, float* dx1, float* dx2, int B, int C1, int C2, int HW, cudaStream_t st) {
    const size_t n1 = size_t(C1) * HW, n2 = size_t(C2) * HW, total = size_t(B) * (n1 + n2);
    concat_bwd_kernel<<<grid_for(total, 256), 256, 0, st>>>(dout, dx1, dx2, total, n1, n2);
}
__global__ void broadcast_fwd_kernel(const float* __restrict__ x, float* __restrict__ out, size_t total, int HW) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x)
        out[i] = x[i / HW];
}
// one warp per row
__global__ void broadcast_bwd_kernel(const float* __restrict__ dout, float* __restrict__ dx, size_t N, int HW) {
    const size_t row = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= N) return;
    float s = 0.f;
    for (int i = lane; i < HW; i += 32) s += dout[row * HW + i];
    for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) dx[row] = s;
}
void broadcast_fwd(const float* x, float* out, size_t N, int HW, cudaStream_t st) {
    const size_t total = N * HW;
    broadcast_fwd_kernel<<<grid_for(total, 256), 256, 0, st>>>(x, out, total, HW);
}
void broadcast_bwd(const float* dout, float* dx, size_t N, int HW, cudaStream_t st) {
    broadcast_bwd_kernel<<<unsigned((N * 32 + 255) / 256), 256, 0, st>>>(dout, dx, N, HW);
}

// ------------------------------------------------------------------------------------------------ loss
__global__ void mse_fwd_kernel(const float* __restrict__ inp, const float* __restrict__ y, float* __restrict__ loss,
                               size_t n, float inv_n) {
    __shared__ float red[32];
    float s = 0.f;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        const float d = inp[i] - y[i];
        s += d * d;
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) atomicAdd(loss, s * inv_n);
}
__global__ void mse_bwd_kernel(const float* __restrict__ inp, const float* __restrict__ y, float* __restrict__ dinp,
                               size_t n, float k) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x)
        dinp[i] = k * (inp[i] - y[i]);
}
void mse_fwd(const float* inp, const float* y, float* loss, size_t n, cudaStream_t st) {
    cudaMemsetAsync(loss, 0, sizeof(float), st);
    mse_fwd_kernel<<<grid_for(n, 256, 2), 256, 0, st>>>(inp, y, loss, n, 1.f / float(n));
}
void mse_bwd(const float* inp, const float* y, float* dinp, size_t n, cudaStream_t st) {
    mse_bwd_kernel<<<grid_for(n, 256), 256, 0, st>>>(inp, y, dinp, n, 2.f / float(n));
}

__global__ void nchw_chansum_kernel(const float* __restrict__ x, int B, int C, size_t HW, float* __restrict__ out) {
    __shared__ float red[32];
    const int c = blockIdx.x;
    float s = 0.f;
    for (int b = 0; b < B; ++b)
        for (size_t i = threadIdx.x; i < HW; i += blockDim.x) s += x[(size_t(b) * C + c) * HW + i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[c] = s;
}
void nchw_chansum(const float* x, int B, int C, size_t HW, float* out, cudaStream_t st) {
    nchw_chansum_kernel<<<C, 256, 0, st>>>(x, B, C, HW, out);
}
__global__ void rows_colsum_kernel(const float* __restrict__ x, int N, int C, float* __restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    float s = 0.f;
    for (int n = 0; n < N; ++n) s += x[size_t(n) * C + c];
    out[c] = s;
}
void rows_colsum(const float* x, int N, int C, float* out, cudaStream_t st) {
    rows_colsum_kernel<<<(C + 127) / 128, 128, 0, st>>>(x, N, C, out);
}

// ------------------------------------------------------------------------------------------------ direct conv
__global__ void conv_direct_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                       const float* __restrict__ b, float* __restrict__ out, size_t total, int Cin,
                                       int Cout, int H, int W, int KS) {
    const int pad = KS / 2, KK = KS * KS;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int ww = int(i % W), h = int((i / W) % H), o = int((i / (size_t(W) * H)) % Cout);
        const size_t bi = i / (size_t(W) * H * Cout);
        float acc = b ? b[o] : 0.f;
        for (int c = 0; c < Cin; ++c) {
            const float* xp = x + (bi * Cin + c) * size_t(H) * W;
            const float* wp = w + (size_t(o) * Cin + c) * KK;
            for (int ky = 0; ky < KS; ++ky) {
                const int hh = h + ky - pad;
                if (hh < 0 || hh >= H) continue;
                for (int kx = 0; kx < KS; ++kx) {
                    const int wx = ww + kx - pad;
                    if (wx < 0 || wx >= W) continue;
                    acc += xp[size_t(hh) * W + wx] * wp[ky * KS + kx];
                }
            }
        }
        out[i] = acc;
    }
}
__global__ void conv_direct_dgrad_kernel(const float* __restrict__ dout, const float* __restrict__ w,
                                         float* __restrict__ dx, size_t total, int Cin, int Cout, int H, int W,
                                         int KS) {
    const int pad = KS / 2, KK = KS * KS;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int ww = int(i % W), h = int((i / W) % H), c = int((i / (size_t(W) * H)) % Cin);
        const size_t bi = i / (size_t(W) * H * Cin);
        float acc = 0.f;
        for (int o = 0; o < Cout; ++o) {
            const float* dp = dout + (bi * Cout + o) * size_t(H) * W;
            const float* wp = w + (size_t(o) * Cin + c) * KK;
            for (int ky = 0; ky < KS; ++ky) {
                const int hh = h - (ky - pad);
                if (hh < 0 || hh >= H) continue;
                for (int kx = 0; kx < KS; ++kx) {
                    const int wx = ww - (kx - pad);
                    if (wx < 0 || wx >= W) continue;
                    acc += dp[size_t(hh) * W + wx] * wp[ky * KS + kx];
                }
            }
        }
        dx[i] = acc;
    }
}
// one block per (o, c): dw[o][c][ky][kx] = sum_{b,h,w} dout[b,o,h,w] * x[b,c,h+ky-pad,w+kx-pad]
__global__ void conv_direct_wgrad_kernel(const float* __restrict__ dout, const float* __restrict__ x,
                                         float* __restrict__ dw, int B, int Cin, int Cout, int H, int W, int KS) {
    __shared__ float red[32];
    const int o = blockIdx.x / Cin, c = blockIdx.x % Cin;
    const int pad = KS / 2, KK = KS * KS;
    float acc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = 0.f;
    const size_t HW = size_t(H) * W;
    for (size_t i = threadIdx.x; i < size_t(B) * HW; i += blockDim.x) {
        const size_t bi = i / HW;
        const int p = int(i % HW), h = p / W, ww = p % W;
        const float d = dout[(bi * Cout + o) * HW + p];
        const float* xp = x + (bi * Cin + c) * HW;
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            if (k < KK) {
                const int hh = h + k / KS - pad, wx = ww + k % KS - pad;
                if (hh >= 0 && hh < H && wx >= 0 && wx < W) acc[k] += d * xp[size_t(hh) * W + wx];
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        if (k < KK) {
            const float s = block_sum(acc[k], red);
            if (threadIdx.x == 0) dw[(size_t(o) * Cin + c) * KK + k] = s;
        }
    }
}
void conv_direct_fwd(const float* x, const float* w, const float* b, float* out, int B, int Cin, int Cout, int H, int W,
                     int KS, cudaStream_t st) {
    const size_t total = size_t(B) * Cout * H * W;
    conv_direct_fwd_kernel<<<grid_for(total, 256, 16), 256, 0, st>>>(x, w, b, out, total, Cin, Cout, H, W, KS);
}
void conv_direct_dgrad(const float* dout, const float* w, float* dx, int B, int Cin, int Cout, int H, int W, int KS,
                       cudaStream_t st) {
    const size_t total = size_t(B) * Cin * H * W;
    conv_direct_dgrad_kernel<<<grid_for(total, 256, 16), 256, 0, st>>>(dout, w, dx, total, Cin, Cout, H, W, KS);
}
void conv_direct_wgrad(const float* dout, const float* x, float* dw, float* db, int B, int Cin, int Cout, int H, int W,
                       int KS, cudaStream_t st) {
    conv_direct_wgrad_kernel<<<Cout * Cin, 256, 0, st>>>(dout, x, dw, B, Cin, Cout, H, W, KS);
    if (db) nchw_chansum(dout, B, Cout, size_t(H) * W, db, st);
}

// ------------------------------------------------------------------------------------------------ attention (fp32)
// inp (B, T, 3, NH, HS) -> qkvr (3, B, NH, T, HS)       (permute_kernel, train_unet.cu:2389)
__global__ void attn_permute_kernel(const float* __restrict__ inp, float* __restrict__ qkvr, size_t total, int B,
                                    int T, int NH, int HS) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int d = int(i % HS), t = int((i / HS) % T), h = int((i / (size_t(HS) * T)) % NH);
        const int b = int((i / (size_t(HS) * T * NH)) % B), s = int(i / (size_t(HS) * T * NH * B));
        qkvr[i] = inp[(((size_t(b) * T + t) * 3 + s) * NH + h) * HS + d];
    }
}
__global__ void attn_unpermute_grad_kernel(const float* __restrict__ dqkvr, float* __restrict__ dinp, size_t total,
                                           int B, int T, int NH, int HS) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int d = int(i % HS), t = int((i / HS) % T), h = int((i / (size_t(HS) * T)) % NH);
        const int b = int((i / (size_t(HS) * T * NH)) % B), s = int(i / (size_t(HS) * T * NH * B));
        dinp[(((size_t(b) * T + t) * 3 + s) * NH + h) * HS + d] = dqkvr[i];
    }
}
// one block per (b, h, t) row: preatt = scale * q.k, att = softmax(preatt)
__global__ void attn_scores_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                   float* __restrict__ preatt, float* __restrict__ att, int T, int HS, float scale) {
    extern __shared__ float srow[];  // [T] + [HS]
    __shared__ float red[32];
    float* sq = srow + T;
    const size_t row = blockIdx.x;        // (b*NH + h)*T + t
    const size_t bh = row / T;
    for (int d = threadIdx.x; d < HS; d += blockDim.x) sq[d] = q[row * HS + d];
    __syncthreads();
    float mx = -INFINITY;
    for (int s = threadIdx.x; s < T; s += blockDim.x) {
        const float* kr = k + (bh * T + s) * HS;
        float a = 0.f;
        for (int d = 0; d < HS; ++d) a += sq[d] * kr[d];
        a *= scale;
        srow[s] = a;
        preatt[row * T + s] = a;
        mx = fmaxf(mx, a);
    }
    for (int off = 16; off; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    mx = red[0];
    for (int i = 1; i < int(blockDim.x >> 5); ++i) mx = fmaxf(mx, red[i]);
    float sum = 0.f;
    for (int s = threadIdx.x; s < T; s += blockDim.x) {
        const float e = expf(srow[s] - mx);
        srow[s] = e;
        sum += e;
    }
    sum = block_sum(sum, red);
    const float inv = 1.f / sum;
    for (int s = threadIdx.x; s < T; s += blockDim.x) att[row * T + s] = srow[s] * inv;
}
// out (B, T, NH, HS) [= (B,T,C)] = att . v ; one thread per output element
__global__ void attn_av_kernel(const float* __restrict__ att, const float* __restrict__ v, float* __restrict__ out,
                               size_t total, int T, int NH, int HS) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int d = int(i % HS), h = int((i / HS) % NH), t = int((i / (size_t(HS) * NH)) % T);
        const size_t b = i / (size_t(HS) * NH * T);
        const size_t bh = b * NH + h;
        const float* ar = att + (bh * T + t) * T;
        const float* vp = v + bh * T * HS + d;
        float a = 0.f;
        for (int s = 0; s < T; ++s) a += ar[s] * vp[size_t(s) * HS];
        out[i] = a;
    }
}
void attention_fwd(float* out, float* qkvr, float* preatt, float* att, const float* inp, int B, int T, int C, int NH,
                   cudaStream_t st) {
    const int HS = C / NH;
    const size_t n = size_t(3) * B * T * C;
    attn_permute_kernel<<<grid_for(n, 256), 256, 0, st>>>(inp, qkvr, n, B, T, NH, HS);
    const float* q = qkvr;
    const float* k = qkvr + size_t(B) * T * C;
    const float* v = qkvr + size_t(2) * B * T * C;
    attn_scores_kernel<<<unsigned(size_t(B) * NH * T), 128, (T + HS) * sizeof(float), st>>>(q, k, preatt, att, T, HS,
                                                                                          1.f / sqrtf(float(HS)));
    const size_t no = size_t(B) * T * C;
    attn_av_kernel<<<grid_for(no, 256, 32), 256, 0, st>>>(att, v, out, no, T, NH, HS);
}
// datt[bh,t,s] = sum_d dout[b,t,h,d] v[bh,s,d] ; dpreatt = att * (datt - sum_s att*datt)   (block per row)
__global__ void attn_bwd_rows_kernel(const float* __restrict__ dout, const float* __restrict__ v,
                                     const float* __restrict__ att, float* __restrict__ datt,
                                     float* __restrict__ dpreatt, int T, int NH, int HS) {
    extern __shared__ float srow[];  // [T] + [HS]
    __shared__ float red[32];
    float* sd = srow + T;
    const size_t row = blockIdx.x;
    const size_t bh = row / T;
    const int t = int(row % T);
    const size_t b = bh / NH;
    const int h = int(bh % NH);
    for (int d = threadIdx.x; d < HS; d += blockDim.x) sd[d] = dout[((b * T + t) * NH + h) * HS + d];
    __syncthreads();
    float dot = 0.f;
    for (int s = threadIdx.x; s < T; s += blockDim.x) {
        const float* vr = v + (bh * T + s) * HS;
        float a = 0.f;
        for (int d = 0; d < HS; ++d) a += sd[d] * vr[d];
        srow[s] = a;
        datt[row * T + s] = a;
        dot += a * att[row * T + s];
    }
    dot = block_sum(dot, red);
    for (int s = threadIdx.x; s < T; s += blockDim.x) dpreatt[row * T + s] = att[row * T + s] * (srow[s] - dot);
}
// dq[bh,t,d] = scale * sum_s dpreatt[t,s] k[s,d] ; dk[bh,s,d] = scale * sum_t dpreatt[t,s] q[t,d] ;
// dv[bh,s,d] = sum_t att[t,s] dout[b,t,h,d]        one thread per (bh, t|s, d)
__global__ void attn_bwd_qkv_kernel(const float* __restrict__ dpreatt, const float* __restrict__ att,
                                    const float* __restrict__ qkvr, const float* __restrict__ dout,
                                    float* __restrict__ dqkvr, size_t per, int B, int T, int NH, int HS,
                                    float scale) {
    const size_t total = per * 3;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += size_t(gridDim.x) * blockDim.x) {
        const int which = int(i / per);
        const size_t r = i % per;
        const int d = int(r % HS), t = int((r / HS) % T);
        const size_t bh = r / (size_t(HS) * T);
        const size_t b = bh / NH;
        const int h = int(bh % NH);
        const float* q = qkvr;
        const float* k = qkvr + per;
        float a = 0.f;
        if (which == 0) {
            const float* pr = dpreatt + (bh * T + t) * T;
            for (int s = 0; s < T; ++s) a += pr[s] * k[(bh * T + s) * HS + d];
            a *= scale;
        } else if (which == 1) {
            for (int tt = 0; tt < T; ++tt) a += dpreatt[(bh * T + tt) * T + t] * q[(bh * T + tt) * HS + d];
            a *= scale;
        } else {
            for (int tt = 0; tt < T; ++tt) a += att[(bh * T + tt) * T + t] * dout[((b * T + tt) * NH + h) * HS + d];
        }
        dqkvr[i] = a;
    }
}
void attention_bwd(float* dinp, float* dqkvr, float* dpreatt, float* datt, const float* dout, const float* qkvr,
                   const float* att, int B, int T, int C, int NH, cudaStream_t st) {
    const int HS = C / NH;
    const size_t per = size_t(B) * T * C;
    const float* v = qkvr + 2 * per;
    attn_bwd_rows_kernel<<<unsigned(size_t(B) * NH * T), 128, (T + HS) * sizeof(float), st>>>(dout, v, att, datt,
                                                                                            dpreatt, T, NH, HS);
    attn_bwd_qkv_kernel<<<grid_for(3 * per, 256, 32), 256, 0, st>>>(dpreatt, att, qkvr, dout, dqkvr, per, B, T, NH, HS,
                                                                   1.f / sqrtf(float(HS)));
    attn_unpermute_grad_kernel<<<grid_for(3 * per, 256), 256, 0, st>>>(dqkvr, dinp, 3 * per, B, T, NH, HS);
}

// ------------------------------------------------------------------------------------------------ small linear
__global__ void linear_fwd_kernel(float* __restrict__ out, const float* __restrict__ inp, const float* __restrict__ w,
                                  const float* __restrict__ b, int N, int C, int OC) {
    const size_t warp = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= size_t(N) * OC) return;
    const size_t n = warp / OC;
    const int o = int(warp % OC);
    float s = 0.f;
    for (int k = lane; k < C; k += 32) s += inp[n * C + k] * w[size_t(o) * C + k];
    for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) out[n * OC + o] = s + (b ? b[o] : 0.f);
}
void linear_fwd(float* out, const float* inp, const float* w, const float* b, int N, int C, int OC, cudaStream_t st) {
    const size_t threads = size_t(N) * OC * 32;
    linear_fwd_kernel<<<unsigned((threads + 255) / 256), 256, 0, st>>>(out, inp, w, b, N, C, OC);
}
__global__ void linear_bwd_w_kernel(float* __restrict__ dw, float* __restrict__ db, const float* __restrict__ dout,
                                    const float* __restrict__ inp, int N, int C, int OC) {
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= size_t(OC) * C) return;
    const int o = int(i / C), k = int(i % C);
    float s = 0.f, sb = 0.f;
    for (int n = 0; n < N; ++n) {
        const float d = dout[size_t(n) * OC + o];
        s += d * inp[size_t(n) * C + k];
        sb += d;
    }
    dw[i] = s;
    if (k == 0 && db) db[o] = sb;
}
__global__ void linear_bwd_x_kernel(float* __restrict__ dinp, const float* __restrict__ dout,
                                    const float* __restrict__ w, int N, int C, int OC) {
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= size_t(N) * C) return;
    const size_t n = i / C;
    const int k = int(i % C);
    float s = 0.f;
    for (int o = 0; o < OC; ++o) s += dout[n * OC + o] * w[size_t(o) * C + k];
    dinp[i] = s;
}
void linear_bwd(float* dinp, float* dw, float* db, const float* dout, const float* inp, const float* w, int N, int C,
                int OC, cudaStream_t st) {
    linear_bwd_w_kernel<<<unsigned((size_t(OC) * C + 255) / 256), 256, 0, st>>>(dw, db, dout, inp, N, C, OC);
    if (dinp) linear_bwd_x_kernel<<<unsigned((size_t(N) * C + 255) / 256), 256, 0, st>>>(dinp, dout, w, N, C, OC);
}

// (B, R, Cc) -> (B, Cc, R) for fp32 matrices, 32x32 tiles through smem: both sides coalesced
__global__ void transpose_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int R, int Cc) {
    __shared__ float t[32][33];
    const size_t base = size_t(blockIdx.z) * R * Cc;
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int r = r0 + i, c = c0 + threadIdx.x;
        if (r < R && c < Cc) t[i][threadIdx.x] = x[base + size_t(r) * Cc + c];
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int c = c0 + i, r = r0 + threadIdx.x;
        if (r < R && c < Cc) y[base + size_t(c) * R + r] = t[threadIdx.x][i];
    }
}
static void transpose_f32(const float* x, float* y, int B, int R, int Cc, cudaStream_t st) {
    dim3 grid((Cc + 31) / 32, (R + 31) / 32, B);
    transpose_f32_kernel<<<grid, dim3(32, 8), 0, st>>>(x, y, R, Cc);
}
void permute_bchw_to_bhwc(const float* x, float* y, int B, int C, int HW, cudaStream_t st) {
    transpose_f32(x, y, B, C, HW, st);
}
void permute_bhwc_to_bchw(const float* x, float* y, int B, int C, int HW, cudaStream_t st) {
    transpose_f32(x, y, B, HW, C, st);
}

}  // namespace f32
}  // namespace ub
