// See misc_ops.cuh.
#include "misc_ops.cuh"
#include <cstdlib>
#include "launch.cuh"

#include <cstdio>

namespace ub {

static constexpr float kLog2e = 1.4426950408889634f;
static constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ void ld8f(const bf16* p, float* f) {
    const uint4 v = *reinterpret_cast<const uint4*>(p);
    const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&u[i]);
        f[2 * i] = __bfloat162float(h.x);
        f[2 * i + 1] = __bfloat162float(h.y);
    }
}
__device__ __forceinline__ void st8f(bf16* p, const float* f) {
    uint32_t u[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
        u[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = make_uint4(u[0], u[1], u[2], u[3]);
}

// =====================================================================================================
// attention core, head size 32 or 64, one row (query for forward / dq, key for dk, dv) per LPR = HS/32 lanes: a lane
// owns 32 channels of its row, and the dot products of a row are combined with one shfl.xor.  (HS = 64 with one thread
// per row would hold 4 x 64 fp32 values per thread in the dkv kernel and spill.)
// =====================================================================================================
static constexpr int kStage = 8192;  // fp32 values of one staged [KT][HS] operand: KT = kStage / HS rows per chunk

// stage `n` rows of an HS-channel slice (row r at src + r*ld) into smem as fp32 [n][HS]
template <int HS>
__device__ __forceinline__ void stage_rows(const bf16* src, int ld, int n, float* dst, float scale) {
    constexpr int kParts = HS / 8, kPartsLog2 = HS == 64 ? 3 : 2;  // 16-byte parts per row
    for (int i = threadIdx.x; i < n * kParts; i += blockDim.x) {
        const int r = i >> kPartsLog2, part = i & (kParts - 1);
        float f[8];
        ld8f(src + size_t(r) * ld + part * 8, f);
#pragma unroll
        for (int k = 0; k < 8; ++k) dst[r * HS + part * 8 + k] = f[k] * scale;
    }
}

// sum of a row's partial dot products over its LPR lanes (adjacent lanes)
template <int LPR>
__device__ __forceinline__ float row_sum(float a) {
    if constexpr (LPR == 2) a += __shfl_xor_sync(0xffffffffu, a, 1);
    return a;
}

// HS = 64 asks for one resident block (minBlocks 1): without that hint ptxas caps the kernel at 96 registers and spills
// the row index across the key loop.  HS = 32 keeps the plain bound (minBlocks 0 = no hint).
template <int HS>
__global__ void __launch_bounds__(128, HS == 64 ? 1 : 0) attn_fwd_kernel(const bf16* __restrict__ qkv, int ld, int T, int NH,
                                                       bf16* __restrict__ out, int ldo, float* __restrict__ lse) {
    constexpr int LPR = HS / 32, KT = kStage / HS;
    pdl_entry();
    extern __shared__ float smf[];  // K [KT][HS], V [KT][HS]
    float* sK = smf;
    float* sV = smf + KT * HS;
    const int h = blockIdx.y, b = blockIdx.z;
    const int C = NH * HS;
    const int part = LPR == 1 ? 0 : int(threadIdx.x) & (LPR - 1);  // this lane's 32 channels: [part*32, part*32+32)
    const int qi = blockIdx.x * (blockDim.x / LPR) + threadIdx.x / LPR;
    const bool active = qi < T;
    const bf16* base = qkv + size_t(b) * T * ld;
    const int ch = h * HS + part * 32;
    float q[32], acc[32];
    const float qscale = rsqrtf(float(HS)) * kLog2e;
    if (active) {
#pragma unroll
        for (int p8 = 0; p8 < 4; ++p8) ld8f(base + size_t(qi) * ld + ch + p8 * 8, q + p8 * 8);
    }
#pragma unroll
    for (int d = 0; d < 32; ++d) q[d] = active ? q[d] * qscale : 0.f, acc[d] = 0.f;
    float m = -1e30f, l = 0.f;
    for (int k0 = 0; k0 < T; k0 += KT) {
        const int nk = min(KT, T - k0);
        __syncthreads();
        stage_rows<HS>(base + size_t(k0) * ld + C + h * HS, ld, nk, sK, 1.f);
        stage_rows<HS>(base + size_t(k0) * ld + 2 * C + h * HS, ld, nk, sV, 1.f);
        __syncthreads();
        for (int j0 = 0; j0 < nk; j0 += 8) {
            float s[8];
            float cmax = -1e30f;
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const float4* kr = reinterpret_cast<const float4*>(sK + (j0 + jj) * HS + part * 32);
                float a = 0.f;
#pragma unroll
                for (int d4 = 0; d4 < 8; ++d4) {
                    const float4 kv = kr[d4];
                    a += q[d4 * 4] * kv.x + q[d4 * 4 + 1] * kv.y + q[d4 * 4 + 2] * kv.z + q[d4 * 4 + 3] * kv.w;
                }
                a = row_sum<LPR>(a);
                s[jj] = (j0 + jj < nk) ? a : -1e30f;
                cmax = fmaxf(cmax, s[jj]);
            }
            if (cmax > m) {
                const float corr = exp2f(m - cmax);
                l *= corr;
#pragma unroll
                for (int d = 0; d < 32; ++d) acc[d] *= corr;
                m = cmax;
            }
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                if (j0 + jj >= nk) continue;  // never touch unstaged smem rows
                const float p = exp2f(s[jj] - m);
                l += p;
                const float4* vr = reinterpret_cast<const float4*>(sV + (j0 + jj) * HS + part * 32);
#pragma unroll
                for (int d4 = 0; d4 < 8; ++d4) {
                    const float4 vv = vr[d4];
                    acc[d4 * 4] += p * vv.x, acc[d4 * 4 + 1] += p * vv.y, acc[d4 * 4 + 2] += p * vv.z,
                        acc[d4 * 4 + 3] += p * vv.w;
                }
            }
        }
    }
    if (active) {
        const float inv = 1.f / l;
#pragma unroll
        for (int d = 0; d < 32; ++d) acc[d] *= inv;
        bf16* op = out + (size_t(b) * T + qi) * ldo + ch;
#pragma unroll
        for (int p8 = 0; p8 < 4; ++p8) st8f(op + p8 * 8, acc + p8 * 8);
        if (part == 0) lse[(size_t(b) * NH + h) * T + qi] = m + log2f(l);
    }
}

// dq: LPR lanes per query
template <int HS>
__global__ void __launch_bounds__(128) attn_bwd_dq_kernel(const bf16* __restrict__ qkv, int ld,
                                                          const bf16* __restrict__ out, int ldo,
                                                          const bf16* __restrict__ dout, int lddo,
                                                          const float* __restrict__ lse, int T, int NH,
                                                          bf16* __restrict__ dqkv, int ldd,
                                                          float* __restrict__ dsum) {
    constexpr int LPR = HS / 32, KT = kStage / HS;
    pdl_entry();
    extern __shared__ float smf[];
    float* sK = smf;
    float* sV = smf + KT * HS;
    const int h = blockIdx.y, b = blockIdx.z;
    const int C = NH * HS;
    const int part = LPR == 1 ? 0 : int(threadIdx.x) & (LPR - 1);
    const int qi = blockIdx.x * (blockDim.x / LPR) + threadIdx.x / LPR;
    const bool active = qi < T;
    const bf16* base = qkv + size_t(b) * T * ld;
    const int ch = h * HS + part * 32;
    float q[32], dO[32], dq[32];
    const float scale = rsqrtf(float(HS));
    float Dv = 0.f, L = 0.f;
    if (active) {
        float o[32];
#pragma unroll
        for (int p8 = 0; p8 < 4; ++p8) {
            ld8f(base + size_t(qi) * ld + ch + p8 * 8, q + p8 * 8);
            ld8f(dout + (size_t(b) * T + qi) * lddo + ch + p8 * 8, dO + p8 * 8);
            ld8f(out + (size_t(b) * T + qi) * ldo + ch + p8 * 8, o + p8 * 8);
        }
#pragma unroll
        for (int d = 0; d < 32; ++d) Dv += dO[d] * o[d];
    }
    Dv = row_sum<LPR>(Dv);  // (both lanes of a row share `active`: the shuffle stays outside the branch)
    if (active) {
        L = lse[(size_t(b) * NH + h) * T + qi];
        if (part == 0) dsum[(size_t(b) * NH + h) * T + qi] = Dv;
    }
#pragma unroll
    for (int d = 0; d < 32; ++d) {
        q[d] = active ? q[d] * scale * kLog2e : 0.f;
        if (!active) dO[d] = 0.f;
        dq[d] = 0.f;
    }
    for (int k0 = 0; k0 < T; k0 += KT) {
        const int nk = min(KT, T - k0);
        __syncthreads();
        stage_rows<HS>(base + size_t(k0) * ld + C + h * HS, ld, nk, sK, 1.f);
        stage_rows<HS>(base + size_t(k0) * ld + 2 * C + h * HS, ld, nk, sV, 1.f);
        __syncthreads();
        for (int j = 0; j < nk; ++j) {
            const float4* kr = reinterpret_cast<const float4*>(sK + j * HS + part * 32);
            const float4* vr = reinterpret_cast<const float4*>(sV + j * HS + part * 32);
            float s = 0.f, dp = 0.f;
#pragma unroll
            for (int d4 = 0; d4 < 8; ++d4) {
                const float4 kv = kr[d4];
                const float4 vv = vr[d4];
                s += q[d4 * 4] * kv.x + q[d4 * 4 + 1] * kv.y + q[d4 * 4 + 2] * kv.z + q[d4 * 4 + 3] * kv.w;
                dp += dO[d4 * 4] * vv.x + dO[d4 * 4 + 1] * vv.y + dO[d4 * 4 + 2] * vv.z + dO[d4 * 4 + 3] * vv.w;
            }
            s = row_sum<LPR>(s), dp = row_sum<LPR>(dp);
            const float ds = exp2f(s - L) * (dp - Dv);
#pragma unroll
            for (int d4 = 0; d4 < 8; ++d4) {
                const float4 kv = kr[d4];
                dq[d4 * 4] += ds * kv.x, dq[d4 * 4 + 1] += ds * kv.y, dq[d4 * 4 + 2] += ds * kv.z,
                    dq[d4 * 4 + 3] += ds * kv.w;
            }
        }
    }
    if (active) {
#pragma unroll
        for (int d = 0; d < 32; ++d) dq[d] *= scale;
        bf16* op = dqkv + (size_t(b) * T + qi) * ldd + ch;
#pragma unroll
        for (int p8 = 0; p8 < 4; ++p8) st8f(op + p8 * 8, dq + p8 * 8);
    }
}

// dk, dv: LPR lanes per key
template <int HS>
__global__ void __launch_bounds__(128) attn_bwd_dkv_kernel(const bf16* __restrict__ qkv, int ld,
                                                           const bf16* __restrict__ dout, int lddo,
                                                           const float* __restrict__ lse,
                                                           const float* __restrict__ dsum, int T, int NH,
                                                           bf16* __restrict__ dqkv, int ldd) {
    constexpr int LPR = HS / 32, KT = kStage / HS;
    pdl_entry();
    extern __shared__ float smf[];  // Q(scaled) [KT][HS], dO [KT][HS], lse [KT], D [KT]
    float* sQ = smf;
    float* sdO = smf + KT * HS;
    float* sL = smf + 2 * KT * HS;
    float* sD = sL + KT;
    const int h = blockIdx.y, b = blockIdx.z;
    const int C = NH * HS;
    const int part = LPR == 1 ? 0 : int(threadIdx.x) & (LPR - 1);
    const int kj = blockIdx.x * (blockDim.x / LPR) + threadIdx.x / LPR;
    const bool active = kj < T;
    const bf16* base = qkv + size_t(b) * T * ld;
    const int ch = h * HS + part * 32;
    float k[32], v[32], dk[32], dv[32];
    if (active) {
#pragma unroll
        for (int p8 = 0; p8 < 4; ++p8) {
            ld8f(base + size_t(kj) * ld + C + ch + p8 * 8, k + p8 * 8);
            ld8f(base + size_t(kj) * ld + 2 * C + ch + p8 * 8, v + p8 * 8);
        }
    }
#pragma unroll
    for (int d = 0; d < 32; ++d) {
        if (!active) k[d] = 0.f, v[d] = 0.f;
        dk[d] = 0.f, dv[d] = 0.f;
    }
    const float qscale = rsqrtf(float(HS)) * kLog2e;
    for (int q0 = 0; q0 < T; q0 += KT) {
        const int nq = min(KT, T - q0);
        __syncthreads();
        stage_rows<HS>(base + size_t(q0) * ld + h * HS, ld, nq, sQ, qscale);
        stage_rows<HS>(dout + (size_t(b) * T + q0) * lddo + h * HS, lddo, nq, sdO, 1.f);
        for (int i = threadIdx.x; i < nq; i += blockDim.x) {
            sL[i] = lse[(size_t(b) * NH + h) * T + q0 + i];
            sD[i] = dsum[(size_t(b) * NH + h) * T + q0 + i];
        }
        __syncthreads();
        for (int i = 0; i < nq; ++i) {
            const float4* qr = reinterpret_cast<const float4*>(sQ + i * HS + part * 32);
            const float4* gr = reinterpret_cast<const float4*>(sdO + i * HS + part * 32);
            float s = 0.f, dp = 0.f;
#pragma unroll
            for (int d4 = 0; d4 < 8; ++d4) {
                const float4 qv = qr[d4];
                const float4 gv = gr[d4];
                s += k[d4 * 4] * qv.x + k[d4 * 4 + 1] * qv.y + k[d4 * 4 + 2] * qv.z + k[d4 * 4 + 3] * qv.w;
                dp += v[d4 * 4] * gv.x + v[d4 * 4 + 1] * gv.y + v[d4 * 4 + 2] * gv.z + v[d4 * 4 + 3] * gv.w;
            }
            s = row_sum<LPR>(s), dp = row_sum<LPR>(dp);
            const float p = exp2f(s - sL[i]);
            const float ds = p * (dp - sD[i]);
#pragma unroll
            for (int d4 = 0; d4 < 8; ++d4) {
                const float4 qv = qr[d4];
                const float4 gv = gr[d4];
                dk[d4 * 4] += ds * qv.x, dk[d4 * 4 + 1] += ds * qv.y, dk[d4 * 4 + 2] += ds * qv.z,
                    dk[d4 * 4 + 3] += ds * qv.w;
                dv[d4 * 4] += p * gv.x, dv[d4 * 4 + 1] += p * gv.y, dv[d4 * 4 + 2] += p * gv.z,
                    dv[d4 * 4 + 3] += p * gv.w;
            }
        }
    }
    if (active) {
        // sQ holds q * scale * log2e, so sum(ds * sQ) = log2e * (scale * sum ds q): multiply by ln2
#pragma unroll
        for (int d = 0; d < 32; ++d) dk[d] *= kLn2;
        bf16* okp = dqkv + (size_t(b) * T + kj) * ldd + C + ch;
        bf16* ovp = dqkv + (size_t(b) * T + kj) * ldd + 2 * C + ch;
#pragma unroll
        for (int p8 = 0; p8 < 4; ++p8) {
            st8f(okp + p8 * 8, dk + p8 * 8);
            st8f(ovp + p8 * 8, dv + p8 * 8);
        }
    }
}

static int attn_block_threads(int T) { return T >= 128 ? 128 : (T >= 64 ? 64 : 32); }
static constexpr int kSmemKV = 2 * kStage * 4;                                        // fwd, dq
template <int HS> static constexpr int smem_attn_dkv() { return (2 * kStage + 2 * (kStage / HS)) * 4; }

void attn_init() {
    static bool cfg = false;
    if (cfg) return;
    cudaFuncSetAttribute(attn_fwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemKV);
    cudaFuncSetAttribute(attn_bwd_dq_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemKV);
    cudaFuncSetAttribute(attn_bwd_dkv_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_attn_dkv<32>());
    cudaFuncSetAttribute(attn_fwd_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemKV);
    cudaFuncSetAttribute(attn_bwd_dq_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemKV);
    cudaFuncSetAttribute(attn_bwd_dkv_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_attn_dkv<64>());
    cfg = true;
}

// grid: (row blocks, NH, B); a block of bt threads covers bt / LPR rows
template <int HS>
static dim3 attn_simt_grid(int B, int T, int NH) {
    const int rows = attn_block_threads(T) / (HS / 32);
    return dim3((T + rows - 1) / rows, NH, B);
}

int attn_fwd(const bf16* qkv, int ld, int B, int T, int NH, int HS, bf16* out, int ldo, float* lse,
             cudaStream_t st) {
    if (HS != 32 && HS != 64) return -20;
    attn_init();
    const int bt = attn_block_threads(T);
    if (HS == 64)
        launch_pdl(attn_fwd_kernel<64>, attn_simt_grid<64>(B, T, NH), dim3(bt), kSmemKV, st, qkv, ld, T, NH, out, ldo, lse);
    else
        launch_pdl(attn_fwd_kernel<32>, attn_simt_grid<32>(B, T, NH), dim3(bt), kSmemKV, st, qkv, ld, T, NH, out, ldo, lse);
    return int(cudaGetLastError());
}

template <int HS>
static void attn_bwd_hs(const bf16* qkv, int ld, const bf16* out, int ldo, const bf16* dout, int lddo, const float* lse,
                        int B, int T, int NH, bf16* dqkv, int ldd, float* dsum, cudaStream_t st) {
    const int bt = attn_block_threads(T);
    const dim3 grid = attn_simt_grid<HS>(B, T, NH);
    launch_pdl(attn_bwd_dq_kernel<HS>, dim3(grid), dim3(bt), kSmemKV, st, qkv, ld, out, ldo, dout, lddo, lse, T, NH, dqkv,
               ldd, dsum);
    launch_pdl(attn_bwd_dkv_kernel<HS>, dim3(grid), dim3(bt), smem_attn_dkv<HS>(), st, qkv, ld, dout, lddo, lse, dsum, T,
               NH, dqkv, ldd);
}

int attn_bwd(const bf16* qkv, int ld, const bf16* out, int ldo, const bf16* dout, int lddo, const float* lse, int B,
             int T, int NH, int HS, bf16* dqkv, int ldd, float* dsum, cudaStream_t st) {
    if (HS != 32 && HS != 64) return -20;
    attn_init();
    if (HS == 64)
        attn_bwd_hs<64>(qkv, ld, out, ldo, dout, lddo, lse, B, T, NH, dqkv, ldd, dsum, st);
    else
        attn_bwd_hs<32>(qkv, ld, out, ldo, dout, lddo, lse, B, T, NH, dqkv, ldd, dsum, st);
    return int(cudaGetLastError());
}

// =====================================================================================================
// small fp32 linears (N = batch rows): one warp per output element, lanes split the reduction
// =====================================================================================================
__device__ __forceinline__ float silu_f(float z) { return z / (1.f + __expf(-z)); }
__device__ __forceinline__ float dsilu_f(float z) {
    const float s = 1.f / (1.f + __expf(-z));
    return s * (1.f + z * (1.f - s));
}

__global__ void small_linear_fwd_kernel(const SmallLinear* __restrict__ table, int N) {
    pdl_entry();
    const SmallLinear e = table[blockIdx.y];
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= N * e.OC) return;
    const int n = warp / e.OC, o = warp % e.OC;
    const float* wr = e.w + size_t(o) * e.C;
    const float* ir = e.inp + size_t(n) * e.C;
    float s = 0.f;
    for (int k = lane; k < e.C; k += 32) {
        float x = ir[k];
        if (e.silu_in) x = silu_f(x);
        s += x * wr[k];
    }
    for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) e.out[size_t(n) * e.OC + o] = s + e.b[o];
}
// Lane = batch row, warp = four output features: the four weight rows are warp-uniform (broadcast) 16-byte loads and
// are read once for 32 batch rows; the activations (N x C fp32, a few KiB) stay in L1.  The warp-per-(row, output)
// kernel above needs N * OC warps per entry -- 22 528 blocks for the 22 embedding projections of a step, i.e. ~19 waves
// of launch overhead for 30 MFLOP; this one is a single wave of 22 x 8 blocks.  C % 4 == 0, OC % 4 == 0.
__global__ void __launch_bounds__(256) small_linear_fwd_rows_kernel(const SmallLinear* __restrict__ table, int N) {
    pdl_entry();
    const SmallLinear e = table[blockIdx.y];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int o = (blockIdx.x * 8 + warp) * 4;
    const int n = blockIdx.z * 32 + lane;
    if (o >= e.OC) return;
    const float4* xr = reinterpret_cast<const float4*>(e.inp + size_t(n < N ? n : N - 1) * e.C);
    const float4* w0 = reinterpret_cast<const float4*>(e.w + size_t(o) * e.C);
    const int C4 = e.C / 4;
    float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8  // (the loads of eight K steps in flight: rolled, every step waited for its own weight rows -- 55 us)
    for (int k = 0; k < C4; ++k) {
        float4 x = __ldg(xr + k);
        if (e.silu_in) x.x = silu_f(x.x), x.y = silu_f(x.y), x.z = silu_f(x.z), x.w = silu_f(x.w);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float4 wv = __ldg(w0 + size_t(u) * C4 + k);
            s[u] = fmaf(x.x, wv.x, s[u]), s[u] = fmaf(x.y, wv.y, s[u]);
            s[u] = fmaf(x.z, wv.z, s[u]), s[u] = fmaf(x.w, wv.w, s[u]);
        }
    }
    if (n < N)
        *reinterpret_cast<float4*>(e.out + size_t(n) * e.OC + o) =
            make_float4(s[0] + e.b[o], s[1] + e.b[o + 1], s[2] + e.b[o + 2], s[3] + e.b[o + 3]);
}
// rows_ok: every entry has C % 4 == 0 and OC % 4 == 0 (the caller knows its table)
void small_linear_fwd(const SmallLinear* table_dev, int n_entries, int N, int max_oc, cudaStream_t st, bool rows_ok) {
    if (rows_ok) {
        launch_pdl(small_linear_fwd_rows_kernel, dim3((max_oc / 4 + 7) / 8, n_entries, (N + 31) / 32), dim3(256), 0, st,
                   table_dev, N);
        return;
    }
    const int warps = N * max_oc;
    launch_pdl(small_linear_fwd_kernel, dim3(dim3((warps * 32 + 255) / 256, n_entries)), dim3(256), 0, st, table_dev, N);
}

// dW[o][k] = sum_n dout[n][o] * act(inp[n][k]) ; db[o] = sum_n dout[n][o]
__global__ void small_linear_bwd_w_kernel(const SmallLinear* __restrict__ table, int N) {
    pdl_entry();
    const SmallLinear e = table[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= e.OC * e.C) return;
    const int o = i / e.C, k = i % e.C;
    float s = 0.f, sb = 0.f;
#pragma unroll 8  // (independent loads: without the unroll the 32 iterations ran back to back at L2 latency each)
    for (int n = 0; n < N; ++n) {
        float x = e.inp[size_t(n) * e.C + k];
        if (e.silu_in) x = silu_f(x);
        const float d = e.dout[size_t(n) * e.OC + o];
        s += d * x;
        sb += d;
    }
    e.dw[i] = s;
    if (k == 0) {
        e.db[o] = sb;
        if (e.db2) e.db2[o] = sb;
    }
}
// dinp[n][k] += sum_o dout[n][o] * W[o][k]; blockIdx.z walks chunks of 32 output channels
__global__ void small_linear_bwd_x_kernel(const SmallLinear* __restrict__ table, int N) {
    pdl_entry();
    const SmallLinear e = table[blockIdx.y];
    if (!e.dinp) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int o0 = blockIdx.z * 32;
    if (i >= N * e.C || o0 >= e.OC) return;
    const int n = i / e.C, k = i % e.C;
    const int o1 = min(o0 + 32, e.OC);
    float s = 0.f;
#pragma unroll 8
    for (int o = o0; o < o1; ++o) s += e.dout[size_t(n) * e.OC + o] * e.w[size_t(o) * e.C + k];
    atomicAdd(&e.dinp[i], s);
}
void small_linear_bwd(const SmallLinear* table_dev, int n_entries, int N, int max_oc, int max_c, cudaStream_t st) {
    launch_pdl(small_linear_bwd_w_kernel, dim3(dim3((max_oc * max_c + 255) / 256, n_entries)), dim3(256), 0, st, table_dev, N);
    launch_pdl(small_linear_bwd_x_kernel, dim3(dim3((N * max_c + 255) / 256, n_entries, (max_oc + 31) / 32)), dim3(256), 0, st, table_dev,
                                                                                                          N);
}

// out[i] = silu(x[i])
__global__ void silu_f32_kernel(const float* __restrict__ x, float* __restrict__ out, size_t n) {
    pdl_entry();
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = silu_f(x[i]);
}
void silu_f32(const float* x, float* out, size_t n, cudaStream_t st) {
    launch_pdl(silu_f32_kernel, dim3(unsigned((n + 255) / 256)), dim3(256), 0, st, x, out, n);
}

__global__ void dsilu_mul_kernel(const float* __restrict__ dact, const float* __restrict__ pre, float* __restrict__ g,
                                 size_t n) {
    pdl_entry();
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) g[i] = dact[i] * dsilu_f(pre[i]);
}
void dsilu_mul(const float* dact, const float* pre, float* g, size_t n, cudaStream_t st) {
    launch_pdl(dsilu_mul_kernel, dim3(unsigned((n + 255) / 256)), dim3(256), 0, st, dact, pre, g, n);
}

__global__ void timestep_embedding_kernel(const float* __restrict__ t, int B, int half, float log_mp,
                                          float* __restrict__ out) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * half) return;
    const int b = i / half, j = i % half;
    const float f = expf(-log_mp * float(j) / float(half));
    const float a = t[b] * f;
    out[size_t(b) * 2 * half + j] = cosf(a);
    out[size_t(b) * 2 * half + half + j] = sinf(a);
}
// The whole time-embedding MLP in one launch (dev/unet.py:176-180, 327-345): sinusoidal embedding -> linear (Cm ->
// Cemb) -> SiLU -> linear (Cemb -> Cemb) -> SiLU, keeping every intermediate the backward pass reads (sin_emb, h0 =
// first pre-activation, emb = second pre-activation, semb = silu(emb)).  Block (b, y) recomputes the first layer of
// batch row b (it is tiny) and produces quarter y of the second layer's outputs.  A warp works on four outputs at a
// time so that their weight rows -- cold in HBM at the start of a step -- are in flight together (one output at a
// time, 16 per warp, measured slower than the four separate launches it replaces).  Same arithmetic and summation
// order per output as timestep_embedding_kernel + small_linear_fwd_kernel + silu_f32_kernel.
constexpr int kTimeMlpSplit = 4;
__device__ __forceinline__ void dot4_rows(const float* __restrict__ x, const float* __restrict__ w, int C, int lane,
                                          float (&s)[4]) {
    s[0] = s[1] = s[2] = s[3] = 0.f;
    for (int k = lane; k < C; k += 32) {
        const float xv = x[k];
#pragma unroll
        for (int u = 0; u < 4; ++u) s[u] += xv * w[size_t(u) * C + k];
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
        for (int off = 16; off; off >>= 1) s[u] += __shfl_xor_sync(0xffffffffu, s[u], off);
}
__global__ void __launch_bounds__(512) time_mlp_fwd_kernel(const float* __restrict__ t, int half, float log_mp,
                                                           const float* __restrict__ w0, const float* __restrict__ b0,
                                                           const float* __restrict__ w1, const float* __restrict__ b1,
                                                           float* __restrict__ sin_emb, float* __restrict__ h0,
                                                           float* __restrict__ emb, float* __restrict__ semb, int Cm,
                                                           int Cemb, const float* __restrict__ label_w,
                                                           const int* __restrict__ labels) {
    pdl_entry();
    extern __shared__ float sm[];
    float* s_in = sm;        // [Cm]
    float* s_h = sm + Cm;    // [Cemb] silu(h0)
    const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const bool writer = blockIdx.y == 0;
    for (int j = threadIdx.x; j < half; j += blockDim.x) {
        const float f = expf(-log_mp * float(j) / float(half));
        const float a = t[b] * f;
        const float c = cosf(a), sn = sinf(a);
        s_in[j] = c, s_in[half + j] = sn;
        if (writer) sin_emb[size_t(b) * Cm + j] = c, sin_emb[size_t(b) * Cm + half + j] = sn;
    }
    __syncthreads();
    for (int o = warp * 4; o < Cemb; o += nwarps * 4) {  // Cemb % 4 == 0
        float s[4];
        dot4_rows(s_in, w0 + size_t(o) * Cm, Cm, lane, s);
        if (lane < 4) {
            const float v = s[lane] + b0[o + lane];
            if (writer) h0[size_t(b) * Cemb + o + lane] = v;
            s_h[o + lane] = silu_f(v);
        }
    }
    __syncthreads();
    const int per = Cemb / kTimeMlpSplit;  // Cemb % 16 == 0
    for (int o = blockIdx.y * per + warp * 4; o < (blockIdx.y + 1) * per; o += nwarps * 4) {
        float s[4];
        dot4_rows(s_h, w1 + size_t(o) * Cemb, Cemb, lane, s);
        if (lane < 4) {
            float v = s[lane] + b1[o + lane];
            // class-conditional model: emb = time_embed(t) + label_emb[y]  (dev/unet.py:301-303)
            if (label_w) v += label_w[size_t(labels[b]) * Cemb + o + lane];
            emb[size_t(b) * Cemb + o + lane] = v;
            semb[size_t(b) * Cemb + o + lane] = silu_f(v);
        }
    }
}
void time_mlp_fwd(const float* t, int B, int Cm, int Cemb, int max_period, const float* w0, const float* b0,
                  const float* w1, const float* b1, float* sin_emb, float* h0, float* emb, float* semb,
                  cudaStream_t st, const float* label_w, const int* labels) {
    launch_pdl(time_mlp_fwd_kernel, dim3(B, kTimeMlpSplit), dim3(512), size_t(Cm + Cemb) * sizeof(float), st, t, Cm / 2,
               logf(float(max_period)), w0, b0, w1, b1, sin_emb, h0, emb, semb, Cm, Cemb, label_w, labels);
}

// d label_emb[y[b]][:] += demb[b][:]  (the backward of the embedding lookup: rows of equal labels add up, hence atomics;
// the gradient arena is zero at the start of a step)
__global__ void label_emb_bwd_kernel(const float* __restrict__ demb, const int* __restrict__ labels, int B, int Cemb,
                                     float* __restrict__ dw) {
    pdl_entry();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * Cemb) return;
    const int b = i / Cemb, j = i - b * Cemb;
    atomicAdd(dw + size_t(labels[b]) * Cemb + j, demb[i]);
}
void label_emb_bwd(const float* demb, const int* labels, int B, int Cemb, float* dw, cudaStream_t st) {
    launch_pdl(label_emb_bwd_kernel, dim3((B * Cemb + 255) / 256), dim3(256), 0, st, demb, labels, B, Cemb, dw);
}

void timestep_embedding(const float* t, int B, int dim, int max_period, float* out, cudaStream_t st) {
    const int half = dim / 2;
    launch_pdl(timestep_embedding_kernel, dim3((B * half + 127) / 128), dim3(128), 0, st, t, B, half, logf(float(max_period)), out);
}

// =====================================================================================================
// diffusion: Philox4x32-10 counter RNG (own implementation; stateless => nothing to checkpoint but seed+step)
// =====================================================================================================
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}
__device__ __forceinline__ float u01(uint32_t x) { return (float(x >> 8) + 0.5f) * (1.f / 16777216.f); }

__global__ void diffusion_t_kernel(int B, int n_timesteps, uint64_t seed, const int* __restrict__ step_dev,
                                   float* __restrict__ t) {
    pdl_entry();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const uint4 r = philox4x32_10(make_uint4(uint32_t(b), 0u, 0x7u, uint32_t(*step_dev)),
                                  make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
    t[b] = float(r.x % uint32_t(n_timesteps));
}
__global__ void diffusion_prepare_kernel(const float* __restrict__ x0, const float* __restrict__ sqrt_ac,
                                         const float* __restrict__ sqrt_1mac, size_t total4, size_t per_image,
                                         uint64_t seed, const int* __restrict__ step_dev, int gen_noise,
                                         const float* __restrict__ t, float* __restrict__ noise,
                                         float* __restrict__ x_t, int W, int* __restrict__ flips) {
    pdl_entry();
    const size_t i4 = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i4 >= total4) return;
    const size_t i = i4 * 4;
    float4 e;
    if (gen_noise) {
        const uint4 r = philox4x32_10(make_uint4(uint32_t(i4), uint32_t(i4 >> 32), 0x1u, uint32_t(*step_dev)),
                                      make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
        const float r0 = sqrtf(-2.f * logf(u01(r.x))), r1 = sqrtf(-2.f * logf(u01(r.z)));
        float s0, c0, s1, c1;
        sincospif(2.f * u01(r.y), &s0, &c0);
        sincospif(2.f * u01(r.w), &s1, &c1);
        e = make_float4(r0 * c0, r0 * s0, r1 * c1, r1 * s1);
        *reinterpret_cast<float4*>(noise + i) = e;
    } else {
        e = *reinterpret_cast<const float4*>(noise + i);
    }
    const int b = int(i / per_image);  // per_image % 4 == 0, so the 4 elements share one image
    const int ti = int(t[b]);
    const float a = sqrt_ac[ti], s = sqrt_1mac[ti];
    float4 x;
    if (flips) {  // random horizontal flip (train_unet.py:531-532), one Philox coin per (step, image); W % 4 == 0
        const uint4 r = philox4x32_10(make_uint4(uint32_t(b), 0u, 0x9u, uint32_t(*step_dev)),
                                      make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
        const int flip = int(r.x >> 31);
        if (i == size_t(b) * per_image) flips[b] = flip;
        if (flip) {
            const size_t row = i - i % size_t(W), w = i % size_t(W);
            const float4 m = *reinterpret_cast<const float4*>(x0 + row + (size_t(W) - 4 - w));
            x = make_float4(m.w, m.z, m.y, m.x);
        } else {
            x = *reinterpret_cast<const float4*>(x0 + i);
        }
    } else {
        x = *reinterpret_cast<const float4*>(x0 + i);
    }
    *reinterpret_cast<float4*>(x_t + i) = make_float4(a * x.x + s * e.x, a * x.y + s * e.y, a * x.z + s * e.z,
                                                      a * x.w + s * e.w);
}
void diffusion_prepare(const float* x0, const float* sqrt_ac, const float* sqrt_1mac, int B, size_t per_image,
                       int n_timesteps, uint64_t seed, const int* step_dev, int gen_t, int gen_noise, float* t,
                       float* noise, float* x_t, cudaStream_t st, int W, int* flips) {
    if (gen_t) launch_pdl(diffusion_t_kernel, dim3((B + 127) / 128), dim3(128), 0, st, B, n_timesteps, seed, step_dev, t);
    const size_t total4 = size_t(B) * per_image / 4;
    launch_pdl(diffusion_prepare_kernel, dim3(unsigned((total4 + 255) / 256)), dim3(256), 0, st, x0, sqrt_ac, sqrt_1mac, total4, per_image,
                                                                             seed, step_dev, gen_noise, t, noise, x_t, W, flips);
}

// classifier-free guidance labels (see misc_ops.cuh); one thread per image
__global__ void cfg_labels_kernel(const int* __restrict__ labels, int* __restrict__ eff, int B, int K, int mode,
                                  float p, uint64_t seed, const int* __restrict__ step_dev) {
    pdl_entry();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int y = mode == CFG_LABELS_NULL ? K : labels[b];
    if (y < 0) y = K;
    if (mode == CFG_LABELS_TRAIN) {
        const uint4 r = philox4x32_10(make_uint4(uint32_t(b), 0u, 0xBu, uint32_t(*step_dev)),
                                      make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
        if (u01(r.x) < p) y = K;
        eff[B + b] = y;
    }
    eff[b] = y;
}
void cfg_labels(const int* labels, int* eff, int B, int K, int mode, float p, uint64_t seed, const int* step_dev,
                cudaStream_t st) {
    launch_pdl(cfg_labels_kernel, dim3((B + 127) / 128), dim3(128), 0, st, labels, eff, B, K, mode, p, seed, step_dev);
}

// Conditioning channels of a super-resolution model (guided-diffusion SuperResModel.forward: F.interpolate(low_res,
// (H, W), mode="bilinear"), align_corners = False).  One block per output row of one (image, channel) plane: the two
// low-res rows the row interpolates between are staged in shared memory, then every output pixel blends four of their
// values.  A low-res pixel is either read from lo (B, C, H/f, W/f) or, in a training step, the f x f area mean of the
// step's image (load_superres_data's F.interpolate(mode="area"), taken from the mirrored image where the step flipped
// it), so the full-resolution image is read about twice rather than 4 f^2 times.  Source coordinates follow torch's
// fp32 arithmetic (area_pixel_compute_source_index, rounded products, no contraction into an FMA).
__device__ __forceinline__ float superres_lowres_px(const float* __restrict__ src, bool full, bool flip, size_t plane,
                                                   int H, int W, int f, int y, int x) {
    if (!full) return __ldg(src + (plane * (H / f) + y) * (W / f) + x);
    float s = 0.f;
    for (int dy = 0; dy < f; ++dy) {
        const float* row = src + (plane * H + size_t(y) * f + dy) * W;
        for (int dx = 0; dx < f; ++dx) s += __ldg(row + (flip ? W - 1 - (x * f + dx) : x * f + dx));
    }
    return s / float(f * f);
}
// torch's source coordinate of output index d (align_corners = False): i0, i1 and the weight of i1
__device__ __forceinline__ void superres_src_index(int d, int n_in, int n_out, int& i0, int& i1, float& l1) {
    const float scale = float(n_in) / float(n_out);
    const float src = fmaxf(__fsub_rn(__fmul_rn(scale, float(d) + 0.5f), 0.5f), 0.f);
    i0 = int(src);
    i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
    l1 = src - float(i0);
}
__global__ void superres_cond_kernel(const float* __restrict__ src, int full, const int* __restrict__ flips, int C,
                                     int H, int W, int f, float* __restrict__ cond) {
    pdl_entry();
    extern __shared__ float srow[];  // [2][W / f]: low-res rows y0, y1
    const int y = blockIdx.x;
    const size_t plane = blockIdx.y;  // b * C + c
    const bool flip = full && flips && flips[plane / C];
    const int hl = H / f, wl = W / f;
    int y0, y1;
    float ly1;
    superres_src_index(y, hl, H, y0, y1, ly1);
    for (int i = threadIdx.x; i < 2 * wl; i += blockDim.x)
        srow[i] = superres_lowres_px(src, full, flip, plane, H, W, f, i < wl ? y0 : y1, i < wl ? i : i - wl);
    __syncthreads();
    const float ly0 = 1.f - ly1;
    float* out = cond + (plane * H + y) * W;
    for (int x = threadIdx.x; x < W; x += blockDim.x) {
        int x0, x1;
        float lx1;
        superres_src_index(x, wl, W, x0, x1, lx1);
        const float lx0 = 1.f - lx1;
        out[x] = ly0 * (lx0 * srow[x0] + lx1 * srow[x1]) + ly1 * (lx0 * srow[wl + x0] + lx1 * srow[wl + x1]);
    }
}
void superres_cond(const float* src, int full, const int* flips, int B, int C, int H, int W, int f, float* cond,
                   cudaStream_t st) {
    launch_pdl(superres_cond_kernel, dim3(unsigned(H), unsigned(B * C)), dim3(128), size_t(2) * (W / f) * sizeof(float),
               st, src, full, flips, C, H, W, f, cond);
}

// =====================================================================================================
// weight packing: 32x32 (o, c) tiles through smem so both packed layouts are written coalesced
// =====================================================================================================
// One 32 (o) x 32 (c) tile of all taps per block.  An o row of the tile is ONE contiguous run of 32 * ntaps floats in
// the (Cout, Cin, taps) master layout: it is read as float4 into raw[oo][cc * ntaps + tap] (row pitch 32 * ntaps + 1
// floats, so that walking oo at fixed (cc, tap) -- the dgrad pack -- and walking cc at fixed (oo, tap) -- stride ntaps,
// odd -- are both bank-conflict free); every thread then writes bf16 PAIRS (4-byte stores, 128 B per warp and row pair).
// (The first version read scalars with a divide per element and wrote 2-byte stores: 31 us per bucket in ncu at 3-6 %
// of the HBM peak; skipping the re-pack bought 0.09 ms of the step, profiles/r02_skip_experiments.txt.)
__global__ void __launch_bounds__(256) pack_weights_kernel(const PackEntry* __restrict__ table) {
    pdl_entry();
    const PackEntry e = table[blockIdx.y];
    const int tiles_c = (e.Cin + 31) / 32, tiles_o = (e.Cout + 31) / 32;
    if (int(blockIdx.x) >= tiles_c * tiles_o) return;
    const int o0 = (blockIdx.x / tiles_c) * 32, c0 = (blockIdx.x % tiles_c) * 32;
    const int nt = e.ntaps;
    const int run = 32 * nt, pitch = run + 1;
    extern __shared__ float raw[];  // [32][pitch]
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 256 threads: ty in 0..7
    const bool full = o0 + 32 <= e.Cout && c0 + 32 <= e.Cin && ((size_t(c0) * nt) % 4) == 0 && ((size_t(e.Cin) * nt) % 4) == 0 &&
                      (reinterpret_cast<uintptr_t>(e.w) & 15) == 0;
    for (int oo = ty; oo < 32; oo += 8) {
        const int o = o0 + oo;
        float* dst = raw + oo * pitch;
        if (full) {
            const float4* src = reinterpret_cast<const float4*>(e.w + (size_t(o) * e.Cin + c0) * nt);
            for (int i = tx; i < run / 4; i += 32) {
                const float4 v = src[i];
                dst[4 * i] = v.x, dst[4 * i + 1] = v.y, dst[4 * i + 2] = v.z, dst[4 * i + 3] = v.w;
            }
        } else {
            for (int i = tx; i < run; i += 32) {
                const int cc = i / nt;
                dst[i] = (o < e.Cout && c0 + cc < e.Cin) ? e.w[(size_t(o) * e.Cin + c0) * nt + i] : 0.f;
            }
        }
    }
    __syncthreads();
    // 16 lanes per 32-element output row (two elements each); a warp writes two rows per step
    const int half = tx >> 4, l2 = (tx & 15) * 2;
    if (e.wf && (e.Cin % 2) == 0) {  // fprop pack [tap][o][c]: rows (tap, oo), pairs along c
        for (int r = ty * 2 + half; r < 32 * nt; r += 16) {
            const int tap = r / 32, oo = r - tap * 32;
            if (o0 + oo < e.Cout && c0 + l2 < e.Cin) {
                const float* sp = raw + oo * pitch + l2 * nt + tap;
                const __nv_bfloat162 v = __floats2bfloat162_rn(sp[0], c0 + l2 + 1 < e.Cin ? sp[nt] : 0.f);
                *reinterpret_cast<__nv_bfloat162*>(e.wf + (size_t(tap) * e.Cout + o0 + oo) * e.Cin + c0 + l2) = v;
            }
        }
    } else if (e.wf) {
        for (int r = ty; r < 32 * nt; r += 8) {
            const int tap = r / 32, oo = r - tap * 32;
            if (o0 + oo < e.Cout && c0 + tx < e.Cin)
                e.wf[(size_t(tap) * e.Cout + o0 + oo) * e.Cin + c0 + tx] = __float2bfloat16(raw[oo * pitch + tx * nt + tap]);
        }
    }
    if (e.wd && (e.Cout % 2) == 0) {  // dgrad pack [ntaps-1-tap][c][o]: rows (tap, cc), pairs along o
        for (int r = ty * 2 + half; r < 32 * nt; r += 16) {
            const int tap = r / 32, cc = r - tap * 32;
            if (c0 + cc < e.Cin && o0 + l2 < e.Cout) {
                const float* sp = raw + l2 * pitch + cc * nt + tap;
                const __nv_bfloat162 v = __floats2bfloat162_rn(sp[0], o0 + l2 + 1 < e.Cout ? sp[pitch] : 0.f);
                *reinterpret_cast<__nv_bfloat162*>(e.wd + (size_t(nt - 1 - tap) * e.Cin + c0 + cc) * e.Cout + o0 + l2) = v;
            }
        }
    } else if (e.wd) {
        for (int r = ty; r < 32 * nt; r += 8) {
            const int tap = r / 32, cc = r - tap * 32;
            if (c0 + cc < e.Cin && o0 + tx < e.Cout)
                e.wd[(size_t(nt - 1 - tap) * e.Cin + c0 + cc) * e.Cout + o0 + tx] =
                    __float2bfloat16(raw[tx * pitch + cc * nt + tap]);
        }
    }
}
void pack_weights(const PackEntry* table_dev, int n_entries, int max_tiles, cudaStream_t st) {
    // (9 taps: 32 x 289 floats = 36 992 B of dynamic shared memory, below the 48 KiB that needs no opt-in)
    launch_pdl(pack_weights_kernel, dim3(dim3(max_tiles, n_entries)), dim3(256), size_t(32) * (32 * 9 + 1) * sizeof(float), st,
               table_dev);
}

// =====================================================================================================
// AdamW
// =====================================================================================================
__global__ void adamw_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, size_t n4, size_t n, float lr, float b1, float b2, float eps,
                             float wd, float gscale, const int* __restrict__ step_dev, const float* __restrict__ hp,
                             float* __restrict__ ema, float ema_rate) {
    pdl_entry();
    // hyper-parameters from device memory when given (the captured step graph: a learning-rate schedule must not force a
    // re-capture), {lr, beta1, beta2, eps, weight_decay}
    if (hp) lr = hp[0], b1 = hp[1], b2 = hp[2], eps = hp[3], wd = hp[4];
    const int t = *step_dev + 1;
    const float c1 = 1.f - powf(b1, float(t)), c2 = 1.f - powf(b2, float(t));
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n4) {
        const float4 pv = reinterpret_cast<float4*>(p)[i], gv = reinterpret_cast<float4*>(g)[i],
                     mv = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
        float pp[4] = {pv.x, pv.y, pv.z, pv.w}, gp[4] = {gv.x, gv.y, gv.z, gv.w}, mp[4] = {mv.x, mv.y, mv.z, mv.w},
              vp[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float gr = gp[k] * gscale;
            mp[k] = b1 * mp[k] + (1.f - b1) * gr;
            vp[k] = b2 * vp[k] + (1.f - b2) * gr * gr;
            const float mh = mp[k] / c1, vh = vp[k] / c2;
            pp[k] -= lr * (mh / (sqrtf(vh) + eps) + wd * pp[k]);
        }
        reinterpret_cast<float4*>(p)[i] = make_float4(pp[0], pp[1], pp[2], pp[3]);
        reinterpret_cast<float4*>(m)[i] = make_float4(mp[0], mp[1], mp[2], mp[3]);
        reinterpret_cast<float4*>(v)[i] = make_float4(vp[0], vp[1], vp[2], vp[3]);
        reinterpret_cast<float4*>(g)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ema) {  // exponential moving average of the updated parameters: ema = rate * ema + (1 - rate) * p
            const float4 ev = reinterpret_cast<float4*>(ema)[i];
            reinterpret_cast<float4*>(ema)[i] =
                make_float4(ema_rate * ev.x + (1.f - ema_rate) * pp[0], ema_rate * ev.y + (1.f - ema_rate) * pp[1],
                            ema_rate * ev.z + (1.f - ema_rate) * pp[2], ema_rate * ev.w + (1.f - ema_rate) * pp[3]);
        }
    } else if (i == n4) {  // tail (n % 4 elements)
        for (size_t k = n4 * 4; k < n; ++k) {
            const float gr = g[k] * gscale;
            m[k] = b1 * m[k] + (1.f - b1) * gr;
            v[k] = b2 * v[k] + (1.f - b2) * gr * gr;
            p[k] -= lr * ((m[k] / c1) / (sqrtf(v[k] / c2) + eps) + wd * p[k]);
            g[k] = 0.f;
            if (ema) ema[k] = ema_rate * ema[k] + (1.f - ema_rate) * p[k];
        }
    }
}
void adamw_step(float* p, float* g, float* m, float* v, size_t n, float lr, float b1, float b2, float eps, float wd,
                float grad_scale, const int* step_dev, cudaStream_t st, const float* hp_dev, float* ema,
                float ema_rate) {
    const size_t n4 = n / 4;
    launch_pdl(adamw_kernel, dim3(unsigned((n4 + 1 + 255) / 256)), dim3(256), 0, st, p, g, m, v, n4, n, lr, b1, b2, eps, wd, grad_scale,
                                                                step_dev, hp_dev, ema, ema_rate);
}
// ---- DDPM sampling
__global__ void sample_set_t_kernel(const int* __restrict__ t_dev, int B, float* __restrict__ tsteps) {
    pdl_entry();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) tsteps[b] = float(*t_dev);
}
void sample_set_t(const int* t_dev, int B, float* tsteps, cudaStream_t st) {
    launch_pdl(sample_set_t_kernel, dim3((B + 127) / 128), dim3(128), 0, st, t_dev, B, tsteps);
}
__device__ __forceinline__ float4 philox_normal4(uint64_t i4, uint32_t stream, uint32_t ctr, uint64_t seed) {
    const uint4 r = philox4x32_10(make_uint4(uint32_t(i4), uint32_t(i4 >> 32), stream, ctr),
                                  make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
    const float r0 = sqrtf(-2.f * logf(u01(r.x))), r1 = sqrtf(-2.f * logf(u01(r.z)));
    float s0, c0, s1, c1;
    sincospif(2.f * u01(r.y), &s0, &c0);
    sincospif(2.f * u01(r.w), &s1, &c1);
    return make_float4(r0 * c0, r0 * s0, r1 * c1, r1 * s1);
}
__global__ void ddpm_step_kernel(float* __restrict__ x, const float* __restrict__ eps, const float* __restrict__ betas,
                                 const float* __restrict__ sqrt_ac, const float* __restrict__ sqrt_1mac,
                                 const float* __restrict__ z, size_t n4, uint64_t seed, const int* __restrict__ t_dev,
                                 const int* __restrict__ it_dev) {
    pdl_entry();
    const size_t i4 = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i4 >= n4) return;
    const int t = *t_dev;  // generate.py: beta_t = betas[t-1], alpha_t = acp[t-1], alpha_t_1 = acp[t-2]
    const float beta = betas[t - 1];
    const float om_t = sqrt_1mac[t - 1] * sqrt_1mac[t - 1], om_t1 = sqrt_1mac[t - 2] * sqrt_1mac[t - 2];
    const float c_eps = beta / sqrt_1mac[t - 1], inv = rsqrtf(1.f - beta), sigma = sqrtf(om_t1 / om_t * beta);
    const float4 xv = reinterpret_cast<const float4*>(x)[i4], ev = reinterpret_cast<const float4*>(eps)[i4];
    const float4 zv = z ? reinterpret_cast<const float4*>(z)[i4] : philox_normal4(i4, 0x3u, uint32_t(*it_dev), seed);
    reinterpret_cast<float4*>(x)[i4] =
        make_float4((xv.x - c_eps * ev.x) * inv + sigma * zv.x, (xv.y - c_eps * ev.y) * inv + sigma * zv.y,
                    (xv.z - c_eps * ev.z) * inv + sigma * zv.z, (xv.w - c_eps * ev.w) * inv + sigma * zv.w);
}
__global__ void sample_advance_kernel(int* t_dev, int* it_dev) {
    pdl_entry();
    *t_dev -= 1;
    *it_dev += 1;
}
void ddpm_step(float* x, const float* eps, const float* betas, const float* sqrt_ac, const float* sqrt_1mac,
               const float* z, size_t n, uint64_t seed, int* t_dev, int* it_dev, cudaStream_t st) {
    const size_t n4 = n / 4;
    launch_pdl(ddpm_step_kernel, dim3(unsigned((n4 + 255) / 256)), dim3(256), 0, st, x, eps, betas, sqrt_ac, sqrt_1mac,
               z, n4, seed, static_cast<const int*>(t_dev), static_cast<const int*>(it_dev));
    launch_pdl(sample_advance_kernel, dim3(1), dim3(1), 0, st, t_dev, it_dev);
}
__global__ void fill_normal_kernel(float* __restrict__ x, size_t n4, uint64_t seed) {
    pdl_entry();
    const size_t i4 = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i4 < n4) reinterpret_cast<float4*>(x)[i4] = philox_normal4(i4, 0x2u, 0u, seed);
}
void fill_normal(float* x, size_t n, uint64_t seed, cudaStream_t st) {
    const size_t n4 = n / 4;
    launch_pdl(fill_normal_kernel, dim3(unsigned((n4 + 255) / 256)), dim3(256), 0, st, x, n4, seed);
}
// ---- respaced sampling
__global__ void spaced_set_t_kernel(const int* __restrict__ ts_table, const SpacedState* __restrict__ s, int B,
                                    float* __restrict__ tsteps) {
    pdl_entry();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) tsteps[b] = float(ts_table[s->it]);
}
void spaced_set_t(const int* ts_table, const SpacedState* s, int B, float* tsteps, cudaStream_t st) {
    launch_pdl(spaced_set_t_kernel, dim3((B + 127) / 128), dim3(128), 0, st, ts_table, s, B, tsteps);
}
// LEARNED (learned-variance model): eps and v are channels 0-2 and 3-5 of the model's (B, 6, H, W) output (img3 = the
// 3 H W floats of one image of x), and sigma = c.sigma * exp(0.5 (frac log beta' + (1 - frac) lpost')) per element,
// frac = (v + 1) / 2, with {log beta', lpost'} in c.pad: c.sigma is the [i > 0] draw flag of the learned-range
// ancestral sampler; DDIM rows leave pad at 0, so that v drops out and sigma is DDIM's.
// GUIDED (classifier-free guidance): eps is the null-class output eps_u, eps_c the conditional output in the same
// layout; eps_u + s (eps_c - eps_u), s = *scale, replaces eps before x0 and the clip, and v is read from eps_c.
template <bool LEARNED, bool GUIDED>
__global__ void spaced_step_kernel(float* __restrict__ x, const float* __restrict__ eps,
                                   const SpacedRow* __restrict__ rows, const float* __restrict__ z, size_t n4,
                                   const SpacedState* __restrict__ s, size_t img3, const float* __restrict__ eps_c,
                                   const float* __restrict__ scale) {
    pdl_entry();
    const size_t i4 = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i4 >= n4) return;
    const int it = s->it;
    const SpacedRow c = rows[it];
    const float4 xv = reinterpret_cast<const float4*>(x)[i4];
    float4 ev, sv = make_float4(c.sigma, c.sigma, c.sigma, c.sigma);
    auto guide = [&](float4 eu, size_t off) {
        if constexpr (GUIDED) {
            const float g = *scale;
            const float4 ec = *reinterpret_cast<const float4*>(eps_c + off);
            eu = make_float4(eu.x + g * (ec.x - eu.x), eu.y + g * (ec.y - eu.y), eu.z + g * (ec.z - eu.z),
                             eu.w + g * (ec.w - eu.w));
        }
        return eu;
    };
    if constexpr (LEARNED) {
        const size_t e = 4 * i4, bi = e / img3, o = bi * 2 * img3 + (e - bi * img3);  // (img3 % 4 == 0)
        ev = guide(*reinterpret_cast<const float4*>(eps + o), o);
        const float4 vv = *reinterpret_cast<const float4*>((GUIDED ? eps_c : eps) + o + img3);
        auto sig = [&](float v) {
            const float frac = 0.5f * (v + 1.f);
            return c.sigma * expf(0.5f * (frac * c.pad[0] + (1.f - frac) * c.pad[1]));
        };
        sv = make_float4(sig(vv.x), sig(vv.y), sig(vv.z), sig(vv.w));
    } else {
        ev = guide(reinterpret_cast<const float4*>(eps)[i4], 4 * i4);
    }
    float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c.sigma != 0.f) zv = z ? reinterpret_cast<const float4*>(z)[i4] : philox_normal4(i4, 0x5u, uint32_t(it), s->seed);
    auto upd = [&](float xs, float es, float zs, float ss) {
        float x0 = c.r * xs - c.rm1 * es;
        if (c.clip != 0.f) x0 = fminf(fmaxf(x0, -1.f), 1.f);
        return c.c_x0 * x0 + c.c_x * xs + ss * zs;
    };
    reinterpret_cast<float4*>(x)[i4] = make_float4(upd(xv.x, ev.x, zv.x, sv.x), upd(xv.y, ev.y, zv.y, sv.y),
                                                   upd(xv.z, ev.z, zv.z, sv.z), upd(xv.w, ev.w, zv.w, sv.w));
}
void spaced_step(float* x, const float* eps, const SpacedRow* rows, const float* z, size_t n, SpacedState* s,
                 cudaStream_t st, size_t img3, const float* eps_c, const float* scale) {
    const size_t n4 = n / 4;
    const dim3 grid(unsigned((n4 + 255) / 256));
    const SpacedState* sc = s;
    auto kernel = eps_c ? (img3 ? spaced_step_kernel<true, true> : spaced_step_kernel<false, true>)
                        : (img3 ? spaced_step_kernel<true, false> : spaced_step_kernel<false, false>);
    launch_pdl(kernel, grid, dim3(256), 0, st, x, eps, rows, z, n4, sc, img3, eps_c, scale);
    increment_step(&s->it, st);
}

// Keeps the stream busy for ~`us` microseconds: the profile replay enqueues a whole step behind it, so the per-op
// CUDA-event intervals measure device time, not how fast the host can submit launches.
__global__ void delay_kernel(unsigned us) {
    const long long t0 = clock64();
    while (clock64() - t0 < (long long)us * 1900) __nanosleep(1000);
}
void stream_delay(unsigned us, cudaStream_t st) { delay_kernel<<<1, 1, 0, st>>>(us); }

__global__ void increment_step_kernel(int* s) {
    pdl_entry(); *s += 1; }
void increment_step(int* step_dev, cudaStream_t st) { launch_pdl(increment_step_kernel, dim3(1), dim3(1), 0, st, step_dev); }

}  // namespace ub
