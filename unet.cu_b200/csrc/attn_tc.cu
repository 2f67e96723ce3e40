// Attention core on the 5th-gen tensor cores (tcgen05 + TMEM), head size 32 or 64, sequence length T <= 256.
//
// Replaces attention_forward1 / attention_backward (/root/reference/train_unet.cu:2553-2760: cuBLAS batched GEMMs
// with materialised (B,NH,T,T) matrices and three permutes) on the internal NHWC bf16 qkv tensor
// [B*T][3C], channel order [Q | K | V], each [NH][HS] (dev/unet.py:75-87).
//
// One CTA = 128 consecutive rows of the flattened (image, position) axis x one 64-channel TMA box (128-byte swizzle)
// of each of Q, K, V.  HS = 32: the box holds a PAIR of heads, a head is selected by the K offset inside the swizzle
// row (+64 B), exactly like a K step of the conv kernels, and the CTA works through the two heads one after the
// other.  HS = 64: the box holds exactly one head (any NH) and the head loop runs once.  All T <= 256 scores of a row
// fit in TMEM, so softmax is exact (no online rescaling).  For T < 128 a tile spans 128/T images and the cross-image
// scores are masked.
//
//   forward : S = Q K^T (K-major x K-major, N = keys) -> TMEM;  row threads: p = exp2(s - max), P (bf16) -> smem in
//             the canonical K-major SW128 layout;  O = P V with V read MN-major straight from its natural layout.
//   dq      : per 128-key chunk  S, dP = dO V^T -> TMEM;  dS = P o (dP - D) -> smem;  dQ += dS K (K MN-major).
//   dkv     : rows are KEYS:  S^T = K Q^T, dP^T = V dO^T -> TMEM;  P^T, dS^T -> smem;  dV += P^T dO, dK += dS^T Q
//             (dO, Q MN-major).  No atomics, no cross-CTA reduction: a CTA owns its 128 keys for all queries.
// The PV-type MMAs use N = 64 (the box's channels of the MN-major operand).  HS = 32 keeps the 32 columns of the
// current head: the wasted half costs 16 tensor cycles per MMA and saves a second descriptor mode.  HS = 64 uses all
// 64.  The score MMAs take K = HS in HS/16 steps of K = 16.
//
// Warp roles: warp 0 = TMA + MMA issue (one elected lane) + TMEM allocator; warps 1-8 = row threads (TMEM lane =
// row; the two warps of a lane quadrant split the columns of every chunk).  mbarriers: load -> s (accumulators ready) -> p (operand written to smem) -> o (second MMA done).
#include "attn_tc.cuh"
#include "igemm.cuh"
#include "launch.cuh"
#include "ptx.cuh"

#include <cstdio>
#include <cstring>

namespace ub {

namespace {

constexpr int kThreads = 288;     // warp 0: TMA + MMA issue; warps 1-8: row threads, two warps per TMEM lane quadrant
constexpr int kRowThreads = 256;  // (the two warps of a quadrant split the columns of every chunk)
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// byte offset of the 16-byte chunk `c16` (0..7) of row r inside a [rows][128 B] SWIZZLE_128B tile
__device__ __forceinline__ uint32_t sw128(int r, int c16) { return uint32_t(r) * 128u + (uint32_t(c16 ^ (r & 7)) << 4); }

// the N = HS/2 accumulator columns a row thread drains per head (HS = 32: 16, HS = 64: 32)
template <int N>
__device__ __forceinline__ void tmem_ld_half(uint32_t taddr, uint32_t (&v)[N]) {
    static_assert(N == 16 || N == 32, "head size 32 or 64");
    if constexpr (N == 16)
        tmem_ld16(taddr, v);
    else
        tmem_ld32(taddr, v);
}

__device__ __forceinline__ uint32_t pack2(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ void unpack8(const uint4& v, float* f) {
    const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&u[i]);
        f[2 * i] = __bfloat162float(h.x), f[2 * i + 1] = __bfloat162float(h.y);
    }
}
// store 32 consecutive columns [col0, col0+32) of row r (bf16) into a K-major SW128 operand made of 16 KiB k-blocks
// of 64 columns
__device__ __forceinline__ void store_row32(uint8_t* tile, int r, int col0, const float (&v)[32]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c8 = col0 / 8 + j;  // 16-byte chunk index along the row
        uint8_t* dst = tile + size_t(c8 >> 3) * 16384 + sw128(r, c8 & 7);
        *reinterpret_cast<uint4*>(dst) = make_uint4(pack2(v[8 * j], v[8 * j + 1]), pack2(v[8 * j + 2], v[8 * j + 3]),
                                                    pack2(v[8 * j + 4], v[8 * j + 5]), pack2(v[8 * j + 6], v[8 * j + 7]));
    }
}

struct Smem {
    uint64_t bar_load, bar_s, bar_p, bar_o;
    uint32_t tmem_slot;
};

// tile geometry shared by the three kernels
struct Tile {
    int row0;    // first row (flattened b*T + t) of the CTA
    int col0;    // first column row (flattened) of the column range
    int ncols;   // columns (keys for fwd/dq, queries for dkv): 128 or 256
    int hp;      // 64-channel box: head pair (HS = 32) or head (HS = 64)
};
__device__ __forceinline__ Tile make_tile(const AttnTcParams& p) {
    Tile t;
    t.row0 = blockIdx.x * 128;
    t.hp = blockIdx.y;
    if (p.T >= 128) {
        t.col0 = (t.row0 / p.T) * p.T;
        t.ncols = p.T;
    } else {
        t.col0 = t.row0;
        t.ncols = 128;
    }
    return t;
}
// column c (tile-local) is visible to row r (tile-local) iff both lie in the same image (T is a power of two);
// MASK is false when a tile lies inside one image (T >= 128)
template <bool MASK>
__device__ __forceinline__ bool same_image(const AttnTcParams& p, int r, int c) {
    if constexpr (MASK) return (r >> p.tshift) == (c >> p.tshift);
    return true;
}

__device__ __forceinline__ void prologue(Smem* sm, uint32_t ncols_tmem, int warp, int lane) {
    if (warp == 0 && lane == 0) {
        mbar_init(&sm->bar_load, 1);
        mbar_init(&sm->bar_s, 1);
        mbar_init(&sm->bar_p, kRowThreads);
        mbar_init(&sm->bar_o, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        tmem_alloc(&sm->tmem_slot, ncols_tmem);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_wait();  // the prologue touched only shared memory and TMEM
}

// =====================================================================================================
// forward
// =====================================================================================================
template <int HS, bool MASK>
__global__ void __launch_bounds__(kThreads) attn_tc_fwd_kernel(const __grid_constant__ AttnTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const Tile t = make_tile(p);
    uint8_t* sQ = smem;                       // [128][128 B]
    uint8_t* sK = sQ + 16384;                 // [ncols][128 B]
    uint8_t* sV = sK + size_t(t.ncols) * 128; // [ncols][128 B]
    uint8_t* sP = sV + size_t(t.ncols) * 128; // [ncols/64][128][128 B]
    float* sx = reinterpret_cast<float*>(sP + size_t(t.ncols) * 256);  // [2 heads][2 halves][128] partial row max
    float* sl = sx + 512;                                              // [2 heads][2 halves][128] partial row sum
    Smem* sm = reinterpret_cast<Smem*>(sl + 512);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int HPB = 64 / HS;  // heads per box
    const int C = p.NH * HS;
    const uint32_t tm_cols = t.ncols > 128 ? 512 : 256;
    const uint32_t o_col = t.ncols;  // O accumulator behind the scores
    // head split (HS = 32 only, see attn_grid): gridDim.z == 2 and the CTA works on ONE head of its pair
    const bool hsplit = HS == 32 && gridDim.z == 2;
    const int h_lo = hsplit ? int(blockIdx.z) : 0, h_hi = hsplit ? int(blockIdx.z) + 1 : HPB;
    prologue(sm, tm_cols, warp, lane);
    const uint32_t tmem = sm->tmem_slot;

    if (warp == 0) {
        // (whole warp converged; TMA / MMA / commit instructions under elect.sync: see elect_one_sync in ptx.cuh)
        {
            const int nbox = t.ncols / 128;
            if (elect_one_sync()) {
                tma_prefetch_desc(&p.tmQKV);
                mbar_expect_tx(&sm->bar_load, uint32_t(16384 * (1 + 2 * nbox)));
                tma_load_2d(sQ, &p.tmQKV, &sm->bar_load, t.hp * 64, t.row0);
                for (int i = 0; i < nbox; ++i) {
                    tma_load_2d(sK + i * 16384, &p.tmQKV, &sm->bar_load, C + t.hp * 64, t.col0 + i * 128);
                    tma_load_2d(sV + i * 16384, &p.tmQKV, &sm->bar_load, 2 * C + t.hp * 64, t.col0 + i * 128);
                }
            }
            __syncwarp();
            mbar_wait(&sm->bar_load, 0);
            tc_fence_after();
            const uint32_t id_s = make_idesc_bf16(128, t.ncols, 0, 0);
            const uint32_t id_o = make_idesc_bf16(128, 64, 0, 1);
            const uint64_t dQ = make_smem_desc_sw128(smem_u32(sQ), 16, 1024), dK = make_smem_desc_sw128(smem_u32(sK), 16, 1024);
            const uint64_t dP = make_smem_desc_sw128(smem_u32(sP), 16, 1024), dV = make_smem_desc_sw128(smem_u32(sV), 8192, 1024);
            for (int h = h_lo; h < h_hi; ++h) {
                if (elect_one_sync()) {
#pragma unroll
                    for (int k = 0; k < HS / 16; ++k)
                        umma_bf16(tmem, dQ + uint64_t(h * (HS / 8) + k * 2), dK + uint64_t(h * (HS / 8) + k * 2), id_s, k);
                    umma_commit(&sm->bar_s);
                }
                __syncwarp();
                mbar_wait(&sm->bar_p, h - h_lo);
                tc_fence_after();
                if (elect_one_sync()) {
#pragma unroll 4
                    for (int j = 0; j < t.ncols / 16; ++j)
                        umma_bf16(tmem + o_col, dP + uint64_t((j >> 2) * 1024 + (j & 3) * 2), dV + uint64_t(j * 128), id_o, j);
                    // (the row threads drain O of the first head before they arrive on bar_p for the second, so its PV may
                    //  reuse the columns)
                    umma_commit(&sm->bar_o);
                }
                __syncwarp();
            }
        }
    } else {
        const int q = warp & 3, half = (warp - 1) >> 2;
        const int r = q * 32 + lane;
        const int gr = t.row0 + r;
        const bool rvalid = gr < p.B * p.T;
        const uint32_t trow = tmem + (uint32_t(q * 32) << 16);
        const float c = rsqrtf(float(HS)) * kLog2e;
        for (int h = h_lo; h < h_hi; ++h) {
            mbar_wait(&sm->bar_s, h - h_lo);
            tc_fence_after();
            float m = -1e30f;
            auto chunk_max = [&](int c0) {
                uint32_t v[32];
                tmem_ld32(trow + c0, v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (same_image<MASK>(p, r, c0 + j)) m = fmaxf(m, __uint_as_float(v[j]));
            };
            if constexpr (HS == 32) {
                for (int c0 = 32 * half; c0 < t.ncols; c0 += 64) chunk_max(c0);
            } else {
                // (without the head loop ptxas unrolls this loop and spills around the overlapping 32-register loads)
#pragma unroll 1
                for (int c0 = 32 * half; c0 < t.ncols; c0 += 64) chunk_max(c0);
            }
            sx[(h * 2 + half) * 128 + r] = m;
            asm volatile("bar.sync 1, 256;" ::: "memory");
            m = fmaxf(m, sx[(h * 2 + (half ^ 1)) * 128 + r]);
            const float mc = m * c;
            float l = 0.f;
            for (int c0 = 32 * half; c0 < t.ncols; c0 += 64) {
                uint32_t v[32];
                tmem_ld32(trow + c0, v);
                tmem_ld_wait();
                float pv[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float e = same_image<MASK>(p, r, c0 + j) ? ex2(fmaf(__uint_as_float(v[j]), c, -mc)) : 0.f;
                    // accumulate the sum of what the tensor core will actually multiply (bf16-rounded)
                    e = __bfloat162float(__float2bfloat16(e));
                    pv[j] = e;
                    l += e;
                }
                store_row32(sP, r, c0, pv);
            }
            sl[(h * 2 + half) * 128 + r] = l;
            fence_async_smem();
            tc_fence_before();
            mbar_arrive(&sm->bar_p);
            mbar_wait(&sm->bar_o, h - h_lo);
            if (h == h_hi - 1) pdl_trigger_late();  // all MMAs of this CTA are complete
            tc_fence_after();
            l += sl[(h * 2 + (half ^ 1)) * 128 + r];  // (ordered by the bar_p arrive / bar_o wait pair)
            uint32_t o[HS / 2];
            tmem_ld_half(trow + o_col + h * HS + half * (HS / 2), o);
            tmem_ld_wait();
            tc_fence_before();
            if (rvalid) {
                const float inv = 1.f / l;
                const int head = t.hp * HPB + h;
                __nv_bfloat16* op = p.out + size_t(gr) * p.ldo + head * HS + half * (HS / 2);
#pragma unroll
                for (int j = 0; j < HS / 16; ++j)
                    reinterpret_cast<uint4*>(op)[j] = make_uint4(
                        pack2(__uint_as_float(o[8 * j]) * inv, __uint_as_float(o[8 * j + 1]) * inv),
                        pack2(__uint_as_float(o[8 * j + 2]) * inv, __uint_as_float(o[8 * j + 3]) * inv),
                        pack2(__uint_as_float(o[8 * j + 4]) * inv, __uint_as_float(o[8 * j + 5]) * inv),
                        pack2(__uint_as_float(o[8 * j + 6]) * inv, __uint_as_float(o[8 * j + 7]) * inv));
                if (half == 0) {
                    const int b = gr / p.T, tt = gr % p.T;
                    p.lse[(size_t(b) * p.NH + head) * p.T + tt] = mc + log2f(l);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, tm_cols);
}

// =====================================================================================================
// backward, dQ (rows = queries)
// =====================================================================================================
template <int HS, bool MASK>
__global__ void __launch_bounds__(kThreads) attn_tc_dq_kernel(const __grid_constant__ AttnTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const Tile t = make_tile(p);
    uint8_t* sQ = smem;
    uint8_t* sdO = sQ + 16384;
    uint8_t* sK = sdO + 16384;
    uint8_t* sV = sK + size_t(t.ncols) * 128;
    uint8_t* sdS = sV + size_t(t.ncols) * 128;  // [2][128][128 B]
    Smem* sm = reinterpret_cast<Smem*>(sdS + 32768);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int HPB = 64 / HS;  // heads per box
    const int C = p.NH * HS;
    prologue(sm, 512, warp, lane);
    const uint32_t tmem = sm->tmem_slot;
    const int nchunk = t.ncols / 128;
    // TMEM columns: S [0,128)  dP [128,256)  dQ_h [256 + 64h, +64)  (HS = 64: one head, dQ [256, 320))

    if (warp == 0) {
        {
            if (elect_one_sync()) {
                tma_prefetch_desc(&p.tmQKV);
                tma_prefetch_desc(&p.tmDO);
                mbar_expect_tx(&sm->bar_load, uint32_t(16384 * (2 + 2 * nchunk)));
                tma_load_2d(sQ, &p.tmQKV, &sm->bar_load, t.hp * 64, t.row0);
                tma_load_2d(sdO, &p.tmDO, &sm->bar_load, t.hp * 64, t.row0);
                for (int i = 0; i < nchunk; ++i) {
                    tma_load_2d(sK + i * 16384, &p.tmQKV, &sm->bar_load, C + t.hp * 64, t.col0 + i * 128);
                    tma_load_2d(sV + i * 16384, &p.tmQKV, &sm->bar_load, 2 * C + t.hp * 64, t.col0 + i * 128);
                }
            }
            __syncwarp();
            mbar_wait(&sm->bar_load, 0);
            tc_fence_after();
            const uint32_t id_s = make_idesc_bf16(128, 128, 0, 0);
            const uint32_t id_o = make_idesc_bf16(128, 64, 0, 1);
            const uint64_t dQ = make_smem_desc_sw128(smem_u32(sQ), 16, 1024), dG = make_smem_desc_sw128(smem_u32(sdO), 16, 1024);
            const uint64_t dK = make_smem_desc_sw128(smem_u32(sK), 16, 1024), dV = make_smem_desc_sw128(smem_u32(sV), 16, 1024);
            const uint64_t dS = make_smem_desc_sw128(smem_u32(sdS), 16, 1024), dKm = make_smem_desc_sw128(smem_u32(sK), 8192, 1024);
            int it = 0;
#pragma unroll 1
            for (int h = 0; h < HPB; ++h) {
                for (int cc = 0; cc < nchunk; ++cc, ++it) {
                    if (elect_one_sync()) {
#pragma unroll
                        for (int k = 0; k < HS / 16; ++k) {
                            const uint64_t o = uint64_t(h * (HS / 8) + k * 2);
                            umma_bf16(tmem, dQ + o, dK + o + uint64_t(cc * 1024), id_s, k);
                            umma_bf16(tmem + 128, dG + o, dV + o + uint64_t(cc * 1024), id_s, k);
                        }
                        umma_commit(&sm->bar_s);
                    }
                    __syncwarp();
                    mbar_wait(&sm->bar_p, it & 1);
                    tc_fence_after();
                    if (elect_one_sync()) {
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            umma_bf16(tmem + 256 + h * 64, dS + uint64_t((j >> 2) * 1024 + (j & 3) * 2),
                                      dKm + uint64_t(cc * 1024 + j * 128), id_o, (cc | j) != 0);
                        umma_commit(&sm->bar_o);
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        const int q = warp & 3, half = (warp - 1) >> 2;
        const int r = q * 32 + lane;
        const int gr = t.row0 + r;
        const bool rvalid = gr < p.B * p.T;
        const uint32_t trow = tmem + (uint32_t(q * 32) << 16);
        const float scale = rsqrtf(float(HS));
        const float c = scale * kLog2e;
        const int b = rvalid ? gr / p.T : 0, tt = rvalid ? gr % p.T : 0;
        // D = rowsum(dO o O), L = logsumexp (log2 domain), per head of the box
        float Dv[2] = {0.f, 0.f}, Lv[2] = {0.f, 0.f};
        if (rvalid) {
#pragma unroll
            for (int h = 0; h < HPB; ++h) {
                const int head = t.hp * HPB + h;
                const uint4* gp = reinterpret_cast<const uint4*>(p.dout + size_t(gr) * p.lddo + head * HS);
                const uint4* op = reinterpret_cast<const uint4*>(p.out + size_t(gr) * p.ldo + head * HS);
                float d = 0.f;
#pragma unroll
                for (int j = 0; j < HS / 8; ++j) {
                    float a[8], o[8];
                    unpack8(gp[j], a);
                    unpack8(op[j], o);
#pragma unroll
                    for (int i = 0; i < 8; ++i) d = fmaf(a[i], o[i], d);
                }
                Dv[h] = d;
                Lv[h] = p.lse[(size_t(b) * p.NH + head) * p.T + tt];
                if (half == 0) p.dsum[(size_t(b) * p.NH + head) * p.T + tt] = d;
            }
        }
        int it = 0;
#pragma unroll 1
        for (int h = 0; h < HPB; ++h) {
            const float Dh = Dv[h], Lh = Lv[h];  // (read once: indexed in the chunk loop they spill)
            for (int cc = 0; cc < nchunk; ++cc, ++it) {
                mbar_wait(&sm->bar_s, it & 1);
                tc_fence_after();
                if (it > 0) mbar_wait(&sm->bar_o, (it - 1) & 1);  // sdS is free again
                for (int c0 = 32 * half; c0 < 128; c0 += 64) {
                    uint32_t s[32], d[32];
                    tmem_ld32(trow + c0, s);
                    tmem_ld32(trow + 128 + c0, d);
                    tmem_ld_wait();
                    float ds[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const bool vis = rvalid && same_image<MASK>(p, r, cc * 128 + c0 + j);
                        const float pr = ex2(fmaf(__uint_as_float(s[j]), c, -Lh));
                        ds[j] = vis ? pr * (__uint_as_float(d[j]) - Dh) : 0.f;
                    }
                    store_row32(sdS, r, c0, ds);
                }
                fence_async_smem();
                tc_fence_before();
                mbar_arrive(&sm->bar_p);
            }
            // dQ of this head is complete when the last chunk's MMAs are
            mbar_wait(&sm->bar_o, (it - 1) & 1);
            if (h == HPB - 1) pdl_trigger_late();  // all MMAs of this CTA are complete
            tc_fence_after();
            uint32_t o[HS / 2];
            tmem_ld_half(trow + 256 + h * 64 + h * HS + half * (HS / 2), o);
            tmem_ld_wait();
            tc_fence_before();
            if (rvalid) {
                __nv_bfloat16* op = p.dqkv + size_t(gr) * p.ldd + (t.hp * HPB + h) * HS + half * (HS / 2);
#pragma unroll
                for (int j = 0; j < HS / 16; ++j)
                    reinterpret_cast<uint4*>(op)[j] = make_uint4(
                        pack2(__uint_as_float(o[8 * j]) * scale, __uint_as_float(o[8 * j + 1]) * scale),
                        pack2(__uint_as_float(o[8 * j + 2]) * scale, __uint_as_float(o[8 * j + 3]) * scale),
                        pack2(__uint_as_float(o[8 * j + 4]) * scale, __uint_as_float(o[8 * j + 5]) * scale),
                        pack2(__uint_as_float(o[8 * j + 6]) * scale, __uint_as_float(o[8 * j + 7]) * scale));
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// =====================================================================================================
// backward, dK and dV (rows = keys, columns = queries)
// =====================================================================================================
template <int HS, bool MASK>
__global__ void __launch_bounds__(kThreads) attn_tc_dkv_kernel(const __grid_constant__ AttnTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const Tile t = make_tile(p);
    uint8_t* sK = smem;                            // rows
    uint8_t* sV = sK + 16384;                      // rows
    uint8_t* sQ = sV + 16384;                      // [ncols][128 B]
    uint8_t* sdO = sQ + size_t(t.ncols) * 128;     // [ncols][128 B]
    uint8_t* sPt = sdO + size_t(t.ncols) * 128;    // [2][128][128 B]
    uint8_t* sdSt = sPt + 32768;                   // [2][128][128 B]
    float* sL = reinterpret_cast<float*>(sdSt + 32768);  // [2 heads][ncols]
    float* sD = sL + 2 * 256;
    Smem* sm = reinterpret_cast<Smem*>(sD + 2 * 256);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int HPB = 64 / HS;  // heads per box
    const int C = p.NH * HS;
    prologue(sm, 512, warp, lane);
    const uint32_t tmem = sm->tmem_slot;
    const int nchunk = t.ncols / 128;
    // TMEM columns: S^T [0,128)  dP^T [128,256)  dK_h [256 + 64h, +64)  dV_h [384 + 64h, +64)
    // (HS = 64: one head, dK [256, 320), dV [384, 448))

    if (warp == 0) {
        {
            if (elect_one_sync()) {
                tma_prefetch_desc(&p.tmQKV);
                tma_prefetch_desc(&p.tmDO);
                mbar_expect_tx(&sm->bar_load, uint32_t(16384 * (2 + 2 * nchunk)));
                tma_load_2d(sK, &p.tmQKV, &sm->bar_load, C + t.hp * 64, t.row0);
                tma_load_2d(sV, &p.tmQKV, &sm->bar_load, 2 * C + t.hp * 64, t.row0);
                for (int i = 0; i < nchunk; ++i) {
                    tma_load_2d(sQ + i * 16384, &p.tmQKV, &sm->bar_load, t.hp * 64, t.col0 + i * 128);
                    tma_load_2d(sdO + i * 16384, &p.tmDO, &sm->bar_load, t.hp * 64, t.col0 + i * 128);
                }
            }
            __syncwarp();
            mbar_wait(&sm->bar_load, 0);
            tc_fence_after();
            const uint32_t id_s = make_idesc_bf16(128, 128, 0, 0);
            const uint32_t id_o = make_idesc_bf16(128, 64, 0, 1);
            const uint64_t dK = make_smem_desc_sw128(smem_u32(sK), 16, 1024), dV = make_smem_desc_sw128(smem_u32(sV), 16, 1024);
            const uint64_t dQ = make_smem_desc_sw128(smem_u32(sQ), 16, 1024), dG = make_smem_desc_sw128(smem_u32(sdO), 16, 1024);
            const uint64_t dPt = make_smem_desc_sw128(smem_u32(sPt), 16, 1024), dSt = make_smem_desc_sw128(smem_u32(sdSt), 16, 1024);
            const uint64_t dQm = make_smem_desc_sw128(smem_u32(sQ), 8192, 1024), dGm = make_smem_desc_sw128(smem_u32(sdO), 8192, 1024);
            int it = 0;
#pragma unroll 1
            for (int h = 0; h < HPB; ++h) {
                for (int cc = 0; cc < nchunk; ++cc, ++it) {
                    if (elect_one_sync()) {
#pragma unroll
                        for (int k = 0; k < HS / 16; ++k) {
                            const uint64_t o = uint64_t(h * (HS / 8) + k * 2);
                            umma_bf16(tmem, dK + o, dQ + o + uint64_t(cc * 1024), id_s, k);
                            umma_bf16(tmem + 128, dV + o, dG + o + uint64_t(cc * 1024), id_s, k);
                        }
                        umma_commit(&sm->bar_s);
                    }
                    __syncwarp();
                    mbar_wait(&sm->bar_p, it & 1);
                    tc_fence_after();
                    if (elect_one_sync()) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const uint64_t aoff = uint64_t((j >> 2) * 1024 + (j & 3) * 2);
                            umma_bf16(tmem + 384 + h * 64, dPt + aoff, dGm + uint64_t(cc * 1024 + j * 128), id_o, (cc | j) != 0);
                            umma_bf16(tmem + 256 + h * 64, dSt + aoff, dQm + uint64_t(cc * 1024 + j * 128), id_o, (cc | j) != 0);
                        }
                        umma_commit(&sm->bar_o);
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        const int q = warp & 3, half = (warp - 1) >> 2;
        const int r = q * 32 + lane;
        const int gr = t.row0 + r;
        const bool rvalid = gr < p.B * p.T;
        const uint32_t trow = tmem + (uint32_t(q * 32) << 16);
        const float scale = rsqrtf(float(HS));
        const float c = scale * kLog2e;
        // logsumexp and D of every query column, every head of the box
        for (int i = threadIdx.x - 32; i < HPB * t.ncols; i += kRowThreads) {
            const int h = i / t.ncols, col = i % t.ncols;
            const int gq = t.col0 + col;
            float L = 0.f, D = 0.f;
            if (gq < p.B * p.T) {
                const int head = t.hp * HPB + h;
                const size_t idx = (size_t(gq / p.T) * p.NH + head) * p.T + gq % p.T;
                L = p.lse[idx];
                // D = rowsum(dO o O) of the query, recomputed here (HS products) instead of read from the dq kernel's
                // dsum: the two backward kernels then have no dependency and run concurrently (attn_tc_bwd)
                const uint4* gp = reinterpret_cast<const uint4*>(p.dout + size_t(gq) * p.lddo + head * HS);
                const uint4* op = reinterpret_cast<const uint4*>(p.out + size_t(gq) * p.ldo + head * HS);
#pragma unroll
                for (int j = 0; j < HS / 8; ++j) {
                    float a[8], o[8];
                    unpack8(gp[j], a);
                    unpack8(op[j], o);
#pragma unroll
                    for (int e = 0; e < 8; ++e) D = fmaf(a[e], o[e], D);
                }
            }
            sL[h * 256 + col] = L, sD[h * 256 + col] = D;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        int it = 0;
#pragma unroll 1
        for (int h = 0; h < HPB; ++h) {
            for (int cc = 0; cc < nchunk; ++cc, ++it) {
                mbar_wait(&sm->bar_s, it & 1);
                tc_fence_after();
                if (it > 0) mbar_wait(&sm->bar_o, (it - 1) & 1);  // sPt / sdSt are free again
                for (int c0 = 32 * half; c0 < 128; c0 += 64) {
                    uint32_t s[32], d[32];
                    tmem_ld32(trow + c0, s);
                    tmem_ld32(trow + 128 + c0, d);
                    tmem_ld_wait();
                    float pt[32], ds[32];
                    const float* Lp = sL + h * 256 + cc * 128 + c0;
                    const float* Dp = sD + h * 256 + cc * 128 + c0;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int col = cc * 128 + c0 + j;
                        const bool vis = rvalid && same_image<MASK>(p, r, col) && (t.col0 + col < p.B * p.T);
                        const float pr = vis ? ex2(fmaf(__uint_as_float(s[j]), c, -Lp[j])) : 0.f;
                        pt[j] = pr;
                        ds[j] = pr * (__uint_as_float(d[j]) - Dp[j]);
                    }
                    store_row32(sPt, r, c0, pt);
                    store_row32(sdSt, r, c0, ds);
                }
                fence_async_smem();
                tc_fence_before();
                mbar_arrive(&sm->bar_p);
            }
            mbar_wait(&sm->bar_o, (it - 1) & 1);
            if (h == HPB - 1) pdl_trigger_late();  // all MMAs of this CTA are complete
            tc_fence_after();
            uint32_t dk[HS / 2], dv[HS / 2];
            tmem_ld_half(trow + 256 + h * 64 + h * HS + half * (HS / 2), dk);
            tmem_ld_half(trow + 384 + h * 64 + h * HS + half * (HS / 2), dv);
            tmem_ld_wait();
            tc_fence_before();
            if (rvalid) {
                __nv_bfloat16* kp = p.dqkv + size_t(gr) * p.ldd + C + (t.hp * HPB + h) * HS + half * (HS / 2);
                __nv_bfloat16* vp = p.dqkv + size_t(gr) * p.ldd + 2 * C + (t.hp * HPB + h) * HS + half * (HS / 2);
#pragma unroll
                for (int j = 0; j < HS / 16; ++j) {
                    reinterpret_cast<uint4*>(kp)[j] = make_uint4(
                        pack2(__uint_as_float(dk[8 * j]) * scale, __uint_as_float(dk[8 * j + 1]) * scale),
                        pack2(__uint_as_float(dk[8 * j + 2]) * scale, __uint_as_float(dk[8 * j + 3]) * scale),
                        pack2(__uint_as_float(dk[8 * j + 4]) * scale, __uint_as_float(dk[8 * j + 5]) * scale),
                        pack2(__uint_as_float(dk[8 * j + 6]) * scale, __uint_as_float(dk[8 * j + 7]) * scale));
                    reinterpret_cast<uint4*>(vp)[j] =
                        make_uint4(pack2(__uint_as_float(dv[8 * j]), __uint_as_float(dv[8 * j + 1])),
                                   pack2(__uint_as_float(dv[8 * j + 2]), __uint_as_float(dv[8 * j + 3])),
                                   pack2(__uint_as_float(dv[8 * j + 4]), __uint_as_float(dv[8 * j + 5])),
                                   pack2(__uint_as_float(dv[8 * j + 6]), __uint_as_float(dv[8 * j + 7])));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

size_t smem_fwd(int ncols) { return 1024 + 16384 + size_t(ncols) * 512 + 4096 + 256; }
size_t smem_dq(int ncols) { return 1024 + 32768 + size_t(ncols) * 256 + 32768 + 256; }
size_t smem_dkv(int ncols) { return 1024 + 32768 + size_t(ncols) * 256 + 65536 + 4096 + 256; }

}  // namespace

// HS = 32 needs an even NH (a 64-channel box holds a pair of heads); HS = 64 takes any NH >= 1
bool attn_tc_supported(int T, int NH, int HS) {
    if (!((HS == 32 && NH >= 2 && NH % 2 == 0) || (HS == 64 && NH >= 1))) return false;
    return T == 256 || T == 128 || T == 64 || T == 32 || T == 16;
}

template <int HS>
static void attn_tc_init_hs() {
    cudaFuncSetAttribute(attn_tc_fwd_kernel<HS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_fwd(256)));
    cudaFuncSetAttribute(attn_tc_dq_kernel<HS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_dq(256)));
    cudaFuncSetAttribute(attn_tc_dkv_kernel<HS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_dkv(256)));
    cudaFuncSetAttribute(attn_tc_fwd_kernel<HS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_fwd(128)));
    cudaFuncSetAttribute(attn_tc_dq_kernel<HS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_dq(128)));
    cudaFuncSetAttribute(attn_tc_dkv_kernel<HS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_dkv(128)));
}

void attn_tc_init() {
    static bool done = false;
    if (done) return;
    attn_tc_init_hs<32>();
    attn_tc_init_hs<64>();
    done = true;
}

int attn_tc_plan(AttnTcParams* p, const __nv_bfloat16* qkv, int ld, int B, int T, int NH, int HS,
                 __nv_bfloat16* out, int ldo, float* lse, const __nv_bfloat16* dout, int lddo, __nv_bfloat16* dqkv,
                 int ldd, float* dsum) {
    memset(p, 0, sizeof(*p));
    if (!attn_tc_supported(T, NH, HS)) return -20;
    const int C = NH * HS;
    if ((ldo % 8) || (ldd % 8) || (lddo % 8)) return -21;
    p->qkv = qkv, p->ld = ld, p->B = B, p->T = T, p->NH = NH, p->HS = HS;
    p->out = out, p->ldo = ldo, p->lse = lse, p->dout = dout, p->lddo = lddo, p->dqkv = dqkv, p->ldd = ldd;
    p->dsum = dsum;
    for (p->tshift = 0; (1 << p->tshift) < T; ++p->tshift) {
    }
    int r = make_bf16_map_2d(&p->tmQKV, qkv, 3 * C, B * T, ld, 128);
    if (r) return r;
    if (dout) r = make_bf16_map_2d(&p->tmDO, dout, C, B * T, lddo, 128);
    return r;
}

// Head split of the forward kernel, HS = 32 only: a CTA owns 128 rows x a PAIR of heads (one 64-channel box); with the
// split the pair is shared by two CTAs (grid z = 2) that each load the box and take one head.  T = 256: 192
// one-per-SM CTAs are two waves on 148 SMs, 384 half CTAs are three half-waves; T = 64: 64 CTAs become 128.  The dq
// and dkv kernels work through both heads of the pair (split: measured, removed, profiles/r02_attn_hsplit.txt).  At
// HS = 64 a box is one head: nothing to split.
static dim3 attn_grid(const AttnTcParams& p, int z) { return dim3((p.B * p.T + 127) / 128, p.NH * p.HS / 64, z); }
static int attn_ncols(const AttnTcParams& p) { return p.T >= 128 ? p.T : 128; }

template <int HS>
static void attn_tc_fwd_hs(const AttnTcParams& p, cudaStream_t st) {
    if (p.T >= 128)
        launch_pdl(attn_tc_fwd_kernel<HS, false>, dim3(attn_grid(p, HS == 32 ? 2 : 1)), dim3(kThreads),
                   smem_fwd(attn_ncols(p)), st, p);
    else
        launch_pdl(attn_tc_fwd_kernel<HS, true>, dim3(attn_grid(p, HS == 32 ? 2 : 1)), dim3(kThreads),
                   smem_fwd(attn_ncols(p)), st, p);
}

int attn_tc_fwd(const AttnTcParams& p, cudaStream_t st) {
    attn_tc_init();
    if (p.HS == 64)
        attn_tc_fwd_hs<64>(p, st);
    else
        attn_tc_fwd_hs<32>(p, st);
    return int(cudaGetLastError());
}

template <int HS>
static void attn_tc_bwd_hs(const AttnTcParams& p, cudaStream_t st, cudaStream_t s2) {
    if (p.T >= 128) {
        launch_pdl(attn_tc_dkv_kernel<HS, false>, dim3(attn_grid(p, 1)), dim3(kThreads), smem_dkv(attn_ncols(p)), s2, p);
        launch_pdl(attn_tc_dq_kernel<HS, false>, dim3(attn_grid(p, 1)), dim3(kThreads), smem_dq(attn_ncols(p)), st, p);
    } else {
        launch_pdl(attn_tc_dkv_kernel<HS, true>, dim3(attn_grid(p, 1)), dim3(kThreads), smem_dkv(attn_ncols(p)), s2, p);
        launch_pdl(attn_tc_dq_kernel<HS, true>, dim3(attn_grid(p, 1)), dim3(kThreads), smem_dq(attn_ncols(p)), st, p);
    }
}

// dq and dkv are independent (each recomputes S and D): with an auxiliary stream and two events the dkv kernel runs
// beside the dq kernel (fork after everything enqueued on st so far, join before st continues); works eagerly and
// under stream capture (the fork / join become graph edges).  aux == nullptr: both on st, one after the other.
int attn_tc_bwd(const AttnTcParams& p, cudaStream_t st, cudaStream_t aux, cudaEvent_t ev_fork, cudaEvent_t ev_join) {
    attn_tc_init();
    cudaStream_t s2 = st;
    if (aux && ev_fork && ev_join) {
        cudaEventRecord(ev_fork, st);
        cudaStreamWaitEvent(aux, ev_fork, 0);
        s2 = aux;
    }
    if (p.HS == 64)
        attn_tc_bwd_hs<64>(p, st, s2);
    else
        attn_tc_bwd_hs<32>(p, st, s2);
    if (s2 != st) {
        cudaEventRecord(ev_join, s2);
        cudaStreamWaitEvent(st, ev_join, 0);
    }
    return int(cudaGetLastError());
}

}  // namespace ub
