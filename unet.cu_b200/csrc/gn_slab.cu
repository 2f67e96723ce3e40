// Single-pass GroupNorm (+SiLU) forward and backward on NHWC bf16 tensors: "slab" kernels.
//
// Replaces groupnorm_forward / groupnorm_backward + silu_forward / silu_backward of the reference
// (/root/reference/train_unet.cu:1768-1991, :305-351: 3 passes over x forward, 3-4 backward, one block per (image, group))
// and this library's own round-1 scheme (statistics accumulated with atomics in the producing conv's epilogue + an apply
// pass): the conv epilogues paid ~0.5 ms per step for the cross-lane column sums (profiles/r02d_ops_nohooks.txt).
//
// One CTA -- or a thread-block cluster of 2/4/8 CTAs splitting the pixels -- owns the slab
//     (image b, channels [c0, c0 + CS)),   CS = lcm(group size, 64 channels) or the whole row,
// i.e. whole normalisation groups of one image and whole 128-byte lines of every pixel row.  Thread t owns the
// 8-channel (16-byte) chunk t % (CS/8) of the pixels pbeg + t / (CS/8) + k * R: consecutive lanes read consecutive 16-byte
// pieces, every request covers full lines (the first version gave a warp 32 pixels x 32 bytes -- one sector per line -- and
// ran at a quarter of the L2 bandwidth).  When its share of the slab fits (K <= 16 vectors per thread forward, 8
// backward) a thread keeps it IN REGISTERS between the statistics and the normalisation, so the tensor is read exactly
// once and written exactly once: 1R + 1W forward, 2R (+1R residual gradient) + 1W backward; larger slabs are read a second
// time (from L2).  No atomics on the statistics, no second kernel, nothing in the conv epilogues.
//
//   reduction : 16 per-thread partial sums (8 channels x {sum, sumsq} / {sum dz, sum dz*xhat}) -> shared memory [16][T],
//               column sums over the R pixel rows of the CTA, then over the cluster through distributed shared memory.
#include "launch.cuh"
#include "nhwc_ops.cuh"

#include <cstdio>

namespace ub {

namespace {

constexpr int kMaxThreads = 512;
constexpr int kMaxCS = 448;  // widest slab: C = 448 (groups of 14 channels: lcm(14, 64) = 448)

struct SlabParams {
    const bf16* x;
    int ldx;
    const bf16* dy;  // backward
    int lddy;
    const bf16* add_in;
    int ldadd;
    bf16* y;  // forward output / backward dx
    int ldy;
    const float* gamma;
    const float* beta;
    float* chsum;   // [B][C][2]: written by forward, read by backward
    float* dgamma;  // backward: += (atomic, one per channel and image)
    float* dbeta;
    float* colsum;  // backward: [B][C] += sum_pix dx (optional)
    int HW, C, cpg, CS, nch8, silu;
    int csz;  // cluster size (CTAs splitting the pixels of a slab)
    int ppc;  // pixels per CTA
    int R;    // pixel rows per sweep = threads / nch8
};

__device__ __forceinline__ void unpack8(const uint4& a, float (&f)[8]) {
    const uint32_t u[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&u[i]);
        f[2 * i] = __bfloat162float(h.x), f[2 * i + 1] = __bfloat162float(h.y);
    }
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
    return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
}
__device__ __forceinline__ float sigmoid_fast(float z) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * z));
    return fmaf(0.5f, t, 0.5f);
}
__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float ld_dsmem(const float* local, uint32_t rank) {
    uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(local)), ra;
    float v;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(rank));
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(ra) : "memory");
    return v;
}

// shared-memory carve-up (floats): scratch[16][T] | tot[16 nch8] | tot2[8 nch8] | full[16 nch8] | 7 x consts[CS]
struct SlabSmem {
    float *scratch, *tot, *tot2, *full, *ca, *cb, *cr, *cm, *cA, *cB, *cC;
    __device__ SlabSmem(float* base, int T, int nch8, int CS) {
        scratch = base, tot = scratch + 16 * T, tot2 = tot + 16 * nch8, full = tot2 + 8 * nch8;
        ca = full + 16 * nch8, cb = ca + CS, cr = cb + CS, cm = cr + CS, cA = cm + CS, cB = cA + CS, cC = cB + CS;
    }
};
size_t slab_smem_bytes(int T, int nch8, int CS) { return sizeof(float) * (size_t(16) * T + 40 * nch8 + 7 * CS); }

// index of (channel c of the slab, statistic st) in tot / full
__device__ __forceinline__ int sidx(int c, int st, int nch8) { return (st * 8 + (c & 7)) * nch8 + (c >> 3); }

// Totals of nval (8 or 16) per-thread values per 8-channel chunk, over the CTA's pixel rows and over the cluster:
// full[j * nch8 + chunk], j < nval.  `tot` is this CTA's partial, read by the cluster peers through DSMEM.
template <int NVAL>
__device__ __forceinline__ void slab_reduce(const SlabParams& p, const float (&mine)[NVAL], float* scratch, float* tot,
                                            float* full) {
    const int T = blockDim.x, t = threadIdx.x;
#pragma unroll
    for (int j = 0; j < NVAL; ++j) scratch[j * T + t] = mine[j];
    __syncthreads();
    // column sums over the R pixel rows: PARTS (a power of two <= 8) consecutive lanes share a value and split the rows,
    // so that all threads work and the dependent chain is R / PARTS loads long (it was R = 64 on 128 threads)
    const int nv = NVAL * p.nch8;
    int parts = 1;
    while (parts < 8 && nv * parts * 2 <= T) parts *= 2;
    for (int v = t / parts; v < ((nv + T / parts - 1) / (T / parts)) * (T / parts); v += T / parts) {  // uniform trip count
        const int part = t % parts;
        float a0 = 0.f, a1 = 0.f;
        if (v < nv) {
            const int j = v / p.nch8, ch = v - j * p.nch8;
            const float* col = scratch + j * T + ch;
            int rr = part;
            for (; rr + parts < p.R; rr += 2 * parts) a0 += col[rr * p.nch8], a1 += col[(rr + parts) * p.nch8];
            if (rr < p.R) a0 += col[rr * p.nch8];
        }
        float a = a0 + a1;
        for (int sft = 1; sft < parts; sft *= 2) a += __shfl_xor_sync(0xffffffffu, a, sft);  // (T % 32 == 0: full warps)
        if (v < nv && part == 0) tot[v] = a;
    }
    if (p.csz > 1) {
        cluster_sync_all();  // every CTA's tot is complete and visible
        for (int v = t; v < nv; v += T) {
            float r8[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) r8[r] = r < p.csz ? ld_dsmem(tot + v, uint32_t(r)) : 0.f;  // 8 loads in flight
            // same order in every CTA of the cluster: bit-identical totals everywhere
            full[v] = ((r8[0] + r8[1]) + (r8[2] + r8[3])) + ((r8[4] + r8[5]) + (r8[6] + r8[7]));
        }
    } else {
        __syncthreads();
        for (int v = t; v < nv; v += T) full[v] = tot[v];
    }
    __syncthreads();
}

// normalisation constants of the slab's channels from per-channel (sum, sumsq) given by `get(c, st)`
template <class Get>
__device__ __forceinline__ void slab_norm_consts(const SlabParams& p, SlabSmem& s, int c0, Get get) {
    const float n = float(p.cpg) * float(p.HW);
    for (int c = threadIdx.x; c < p.CS; c += blockDim.x) {
        const int g0 = (c / p.cpg) * p.cpg;
        float su = 0.f, sq = 0.f;
        for (int k = 0; k < p.cpg; ++k) su += get(g0 + k, 0), sq += get(g0 + k, 1);
        const float mean = su / n;
        const float var = fmaxf(sq / n - mean * mean, 0.f);
        const float r = rsqrtf(var + 1e-5f);
        const float a = r * p.gamma[c0 + c];
        s.cr[c] = r, s.cm[c] = mean * r, s.ca[c] = a, s.cb[c] = p.beta[c0 + c] - mean * a;
    }
}

struct SlabGeom {
    int b, c0, chunk, r, pbeg, pend;
    size_t img;
};
__device__ __forceinline__ SlabGeom slab_geom(const SlabParams& p, uint32_t rank) {
    SlabGeom g;
    g.b = blockIdx.y;
    g.c0 = (blockIdx.x / p.csz) * p.CS;
    g.r = threadIdx.x / p.nch8, g.chunk = threadIdx.x - g.r * p.nch8;
    g.pbeg = int(rank) * p.ppc, g.pend = min(g.pbeg + p.ppc, p.HW);
    g.img = size_t(g.b) * p.HW;
    return g;
}

// ------------------------------------------------------------------------------------------------ forward
// K > 0: the thread's K vectors stay in registers between the two phases; K == 0: loop mode (second read from L2)
template <int K>
__global__ void __launch_bounds__(kMaxThreads) gn_slab_fwd_kernel(const SlabParams p) {
    pdl_entry();
    extern __shared__ float slab_sm[];
    SlabSmem s(slab_sm, blockDim.x, p.nch8, p.CS);
    const uint32_t rank = p.csz > 1 ? cluster_rank() : 0u;
    const SlabGeom g = slab_geom(p, rank);
    const bf16* xp = p.x + g.c0 + g.chunk * 8;
    bf16* yp = p.y + g.c0 + g.chunk * 8;
    constexpr int KR = K > 0 ? K : 1;
    uint4 v[KR];
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    auto accumulate = [&](const uint4& u) {
        float f[8];
        unpack8(u, f);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] += f[i], acc[8 + i] = fmaf(f[i], f[i], acc[8 + i]);
    };
    if constexpr (K > 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int pix = g.pbeg + k * p.R + g.r;
            v[k] = pix < g.pend ? *reinterpret_cast<const uint4*>(xp + (g.img + pix) * p.ldx) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) accumulate(v[k]);
    } else {
        for (int pix = g.pbeg + g.r; pix < g.pend; pix += 4 * p.R) {
            uint4 u[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int pp = pix + j * p.R;
                u[j] = pp < g.pend ? *reinterpret_cast<const uint4*>(xp + (g.img + pp) * p.ldx) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) accumulate(u[j]);
        }
    }
    slab_reduce<16>(p, acc, s.scratch, s.tot, s.full);
    if (rank == 0)  // the backward pass reads chsum[B][C][2]
        for (int c = threadIdx.x; c < p.CS; c += blockDim.x)
            *reinterpret_cast<float2*>(p.chsum + (size_t(g.b) * p.C + g.c0 + c) * 2) =
                make_float2(s.full[sidx(c, 0, p.nch8)], s.full[sidx(c, 1, p.nch8)]);
    slab_norm_consts(p, s, g.c0, [&](int c, int st) { return s.full[sidx(c, st, p.nch8)]; });
    __syncthreads();
    float a[8], bb[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = s.ca[g.chunk * 8 + i], bb[i] = s.cb[g.chunk * 8 + i];
    auto apply = [&](const uint4& u, int pix) {
        float f[8];
        unpack8(u, f);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float z = fmaf(f[i], a[i], bb[i]);
            f[i] = p.silu ? z * sigmoid_fast(z) : z;
        }
        *reinterpret_cast<uint4*>(yp + (g.img + pix) * p.ldy) = pack8(f);
    };
    if constexpr (K > 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int pix = g.pbeg + k * p.R + g.r;
            if (pix < g.pend) apply(v[k], pix);
        }
    } else {
        for (int pix = g.pbeg + g.r; pix < g.pend; pix += 4 * p.R) {
            uint4 u[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int pp = pix + j * p.R;
                u[j] = pp < g.pend ? *reinterpret_cast<const uint4*>(xp + (g.img + pp) * p.ldx) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (pix + j * p.R < g.pend) apply(u[j], pix + j * p.R);
        }
    }
    if (p.csz > 1) cluster_sync_all();  // peers may still be reading this CTA's totals
}

// ------------------------------------------------------------------------------------------------ backward
// dy = dL/d act(gn(x)) with act = SiLU (silu = 1) or identity (silu = 0).
//   dz = dy * act'(z)   (rounded to bf16)                             S1_c = sum_p dz,  S2_c = sum_p dz * xhat
//   dgamma_c += S2_c, dbeta_c += S1_c;   per group: m1 = sum_c gamma_c S1_c, m2 = sum_c gamma_c S2_c
//   dx = rstd * (gamma*dz - m1/n - xhat*m2/n) [+ add_in]             colsum[b][c] += sum_p (dx without add_in)
template <int K>
__global__ void __launch_bounds__(kMaxThreads) gn_slab_bwd_kernel(const SlabParams p) {
    pdl_entry();
    extern __shared__ float slab_sm[];
    SlabSmem s(slab_sm, blockDim.x, p.nch8, p.CS);
    const uint32_t rank = p.csz > 1 ? cluster_rank() : 0u;
    const SlabGeom g = slab_geom(p, rank);
    const bf16* xp = p.x + g.c0 + g.chunk * 8;
    const bf16* dp = p.dy + g.c0 + g.chunk * 8;
    constexpr int KR = K > 0 ? K : 1;
    uint4 vx[KR], vd[KR];
    if constexpr (K > 0) {  // issue the loads before the (global-memory dependent) constants are computed
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int pix = g.pbeg + k * p.R + g.r;
            const bool ok = pix < g.pend;
            vx[k] = ok ? *reinterpret_cast<const uint4*>(xp + (g.img + pix) * p.ldx) : make_uint4(0, 0, 0, 0);
            vd[k] = ok ? *reinterpret_cast<const uint4*>(dp + (g.img + pix) * p.lddy) : make_uint4(0, 0, 0, 0);
        }
    }
    {
        const float* cs_b = p.chsum + (size_t(g.b) * p.C + g.c0) * 2;
        slab_norm_consts(p, s, g.c0, [&](int c, int st) { return cs_b[c * 2 + st]; });
    }
    __syncthreads();
    float ca[8], cb[8], cr[8], cm[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = g.chunk * 8 + i;
        ca[i] = s.ca[c], cb[i] = s.cb[c], cr[i] = s.cr[c], cm[i] = s.cm[c];
    }
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    // dz (bf16-rounded, packed) of one vector; accumulates S1 / S2 of exactly the rounded values
    auto dz_of = [&](const uint4& ux, const uint4& ud, bool accumulate) -> uint4 {
        float f[8], d[8];
        unpack8(ux, f);
        unpack8(ud, d);
        if (p.silu) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float z = fmaf(f[i], ca[i], cb[i]);
                const float sg = sigmoid_fast(z);
                d[i] *= sg * fmaf(z, 1.f - sg, 1.f);
            }
        }
        const uint4 o = pack8(d);
        if (accumulate) {
            float dr[8];
            unpack8(o, dr);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] += dr[i], acc[8 + i] = fmaf(dr[i], fmaf(f[i], cr[i], -cm[i]), acc[8 + i]);
        }
        return o;
    };
    if constexpr (K > 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) vd[k] = dz_of(vx[k], vd[k], true);  // zero vectors outside the slab add nothing
    } else {
        for (int pix = g.pbeg + g.r; pix < g.pend; pix += 2 * p.R) {
            uint4 ux[2], ud[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int pp = pix + j * p.R;
                const bool ok = pp < g.pend;
                ux[j] = ok ? *reinterpret_cast<const uint4*>(xp + (g.img + pp) * p.ldx) : make_uint4(0, 0, 0, 0);
                ud[j] = ok ? *reinterpret_cast<const uint4*>(dp + (g.img + pp) * p.lddy) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) dz_of(ux[j], ud[j], true);
        }
    }
    slab_reduce<16>(p, acc, s.scratch, s.tot, s.full);
    {
        const float n = float(p.cpg) * float(p.HW);
        for (int c = threadIdx.x; c < p.CS; c += blockDim.x) {
            const int g0 = (c / p.cpg) * p.cpg;
            float m1 = 0.f, m2 = 0.f;
            for (int k = 0; k < p.cpg; ++k) {
                const float gm = p.gamma[g.c0 + g0 + k];
                m1 = fmaf(gm, s.full[sidx(g0 + k, 0, p.nch8)], m1);
                m2 = fmaf(gm, s.full[sidx(g0 + k, 1, p.nch8)], m2);
            }
            const float r = s.cr[c];
            const float c1 = r * m1 / n, c2 = r * m2 / n;
            s.cA[c] = s.ca[c], s.cB[c] = c2 * r, s.cC[c] = s.cm[c] * c2 - c1;
            if (rank == 0) {
                atomicAdd(p.dgamma + g.c0 + c, s.full[sidx(c, 1, p.nch8)]);
                atomicAdd(p.dbeta + g.c0 + c, s.full[sidx(c, 0, p.nch8)]);
            }
        }
    }
    __syncthreads();
    float cA[8], cB[8], cC[8], csum[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = g.chunk * 8 + i;
        cA[i] = s.cA[c], cB[i] = s.cB[c], cC[i] = s.cC[c], csum[i] = 0.f;
    }
    bf16* op = p.y + g.c0 + g.chunk * 8;
    const bf16* ap = p.add_in ? p.add_in + g.c0 + g.chunk * 8 : nullptr;
    auto apply = [&](const uint4& ux, const uint4& udz, int pix) {
        float f[8], d[8], a[8];
        unpack8(ux, f);
        unpack8(udz, d);
        if (ap) {
            unpack8(*reinterpret_cast<const uint4*>(ap + (g.img + pix) * p.ldadd), a);
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = 0.f;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float gg = fmaf(cA[i], d[i], fmaf(-cB[i], f[i], cC[i]));
            csum[i] += gg;
            a[i] += gg;
        }
        *reinterpret_cast<uint4*>(op + (g.img + pix) * p.ldy) = pack8(a);
    };
    if constexpr (K > 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int pix = g.pbeg + k * p.R + g.r;
            if (pix < g.pend) apply(vx[k], vd[k], pix);
        }
    } else {
        for (int pix = g.pbeg + g.r; pix < g.pend; pix += 2 * p.R) {
            uint4 ux[2], ud[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int pp = pix + j * p.R;
                const bool ok = pp < g.pend;
                ux[j] = ok ? *reinterpret_cast<const uint4*>(xp + (g.img + pp) * p.ldx) : make_uint4(0, 0, 0, 0);
                ud[j] = ok ? *reinterpret_cast<const uint4*>(dp + (g.img + pp) * p.lddy) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int j = 0; j < 2; ++j)
                if (pix + j * p.R < g.pend) apply(ux[j], dz_of(ux[j], ud[j], false), pix + j * p.R);
        }
    }
    if (p.colsum) {  // per-image column sums of dx (embedding-projection backward)
        slab_reduce<8>(p, csum, s.scratch, s.tot2, s.full);
        if (rank == 0)
            for (int c = threadIdx.x; c < p.CS; c += blockDim.x)
                atomicAdd(p.colsum + size_t(g.b) * p.C + g.c0 + c, s.full[sidx(c, 0, p.nch8)]);
    }
    if (p.csz > 1) cluster_sync_all();
}

// ------------------------------------------------------------------------------------------------ planning
struct SlabPlan {
    int CS, nch8, threads, R, K, csz, ppc;  // K == 0: loop mode
};
int gcd(int a, int b) { return b ? gcd(b, a % b) : a; }

bool slab_plan(int B, int HW, int C, int G, bool backward, SlabPlan* pl) {
    if (G < 1 || C % G || C % 8 || HW < 1) return false;
    const int cpg = C / G;
    int CS = cpg / gcd(cpg, 64) * 64;  // lcm(group size, 64 channels = one 128-byte line)
    if (CS > C || C % CS) CS = C;      // otherwise whole rows
    if (CS > kMaxCS || CS % cpg) return false;
    const int nch8 = CS / 8;
    const int slabs = B * (C / CS);
    // cluster size: the smallest that puts >= 256 CTAs on the chip (or the largest, 8)
    int csz = 1;
    while (csz < 8 && slabs * csz < 256 && (HW + 2 * csz - 1) / (2 * csz) >= 4) csz *= 2;
    const int ppc = (HW + csz - 1) / csz;
    // pixel rows per sweep: threads = nch8 * R must be a multiple of 32 and <= 512; no more rows than pixels
    const int rstep = 32 / gcd(nch8, 32);
    int R = (kMaxThreads / nch8) / rstep * rstep;
    while (R > rstep && R - rstep >= ppc) R -= rstep;
    if (R < rstep) return false;
    int need = (ppc + R - 1) / R, K = 1;
    while (K < need) K *= 2;
    if (K > (backward ? 8 : 16)) K = 0;  // does not fit the registers: loop mode
    *pl = SlabPlan{CS, nch8, nch8 * R, R, K, csz, ppc};
    return true;
}

template <int K>
void launch_slab(bool fwd, const SlabParams& p, dim3 grid, int threads, cudaStream_t st) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = dim3(threads), cfg.stream = st;
    cfg.dynamicSmemBytes = slab_smem_bytes(threads, p.nch8, p.CS);
    cudaLaunchAttribute at[2];
    int n = 0;
    if (pdl_enabled()) {
        at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (p.csz > 1) {
        at[n].id = cudaLaunchAttributeClusterDimension;
        at[n].val.clusterDim.x = unsigned(p.csz), at[n].val.clusterDim.y = 1, at[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = at, cfg.numAttrs = n;
    cudaError_t e = fwd ? cudaLaunchKernelEx(&cfg, gn_slab_fwd_kernel<K>, p) : cudaLaunchKernelEx(&cfg, gn_slab_bwd_kernel<K>, p);
    if (e != cudaSuccess)
        fprintf(stderr, "[unet_b200] gn_slab launch failed: %s (grid %u x %u, %d threads, cluster %d, K %d)\n",
                cudaGetErrorString(e), grid.x, grid.y, threads, p.csz, K);
}

template <int K>
void slab_attr() {
    const int mx = int(slab_smem_bytes(kMaxThreads, kMaxCS / 8, kMaxCS));
    cudaFuncSetAttribute(gn_slab_fwd_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    cudaFuncSetAttribute(gn_slab_bwd_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
}

bool aligned_ok(const void* ptr, int ld) { return (reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && ld % 8 == 0; }

void fill_geom(SlabParams& p, const SlabPlan& pl, int HW, int C, int G, int silu) {
    p.HW = HW, p.C = C, p.cpg = C / G, p.CS = pl.CS, p.nch8 = pl.nch8, p.silu = silu, p.csz = pl.csz, p.ppc = pl.ppc;
    p.R = pl.R;
}

}  // namespace

// opt-in shared memory (the [16][T] reduction scratch exceeds 48 KiB at 512 threads); call before graph capture
void gn_slab_init() {
    static bool done = false;
    if (done) return;
    slab_attr<0>(), slab_attr<1>(), slab_attr<2>(), slab_attr<4>(), slab_attr<8>(), slab_attr<16>();
    done = true;
}

bool gn_slab_supported(int B, int HW, int C, int G, bool backward) {
    SlabPlan pl;
    return slab_plan(B, HW, C, G, backward, &pl);
}

int gn_slab_fwd(const bf16* x, int ldx, const float* gamma, const float* beta, int B, int HW, int C, int G, int silu,
                bf16* y, int ldy, float* chsum, cudaStream_t st) {
    SlabPlan pl;
    if (!slab_plan(B, HW, C, G, false, &pl) || !aligned_ok(x, ldx) || !aligned_ok(y, ldy)) return -1;
    gn_slab_init();
    SlabParams p{};
    p.x = x, p.ldx = ldx, p.y = y, p.ldy = ldy, p.gamma = gamma, p.beta = beta, p.chsum = chsum;
    fill_geom(p, pl, HW, C, G, silu);
    const dim3 grid(unsigned(C / pl.CS * pl.csz), unsigned(B));
    switch (pl.K) {
        case 0: launch_slab<0>(true, p, grid, pl.threads, st); break;
        case 1: launch_slab<1>(true, p, grid, pl.threads, st); break;
        case 2: launch_slab<2>(true, p, grid, pl.threads, st); break;
        case 4: launch_slab<4>(true, p, grid, pl.threads, st); break;
        case 8: launch_slab<8>(true, p, grid, pl.threads, st); break;
        default: launch_slab<16>(true, p, grid, pl.threads, st); break;
    }
    return 0;
}

int gn_slab_bwd(const bf16* x, int ldx, const bf16* dy, int lddy, const float* chsum, const float* gamma,
                const float* beta, int B, int HW, int C, int G, int silu, const bf16* add_in, int ldadd, bf16* dx,
                int lddx, float* dgamma, float* dbeta, float* colsum_out, cudaStream_t st) {
    SlabPlan pl;
    if (!slab_plan(B, HW, C, G, true, &pl) || !aligned_ok(x, ldx) || !aligned_ok(dy, lddy) || !aligned_ok(dx, lddx) ||
        (add_in && !aligned_ok(add_in, ldadd)))
        return -1;
    gn_slab_init();
    SlabParams p{};
    p.x = x, p.ldx = ldx, p.dy = dy, p.lddy = lddy, p.add_in = add_in, p.ldadd = ldadd, p.y = dx, p.ldy = lddx;
    p.gamma = gamma, p.beta = beta, p.chsum = const_cast<float*>(chsum), p.dgamma = dgamma, p.dbeta = dbeta;
    p.colsum = colsum_out;
    fill_geom(p, pl, HW, C, G, silu);
    const dim3 grid(unsigned(C / pl.CS * pl.csz), unsigned(B));
    switch (pl.K) {
        case 0: launch_slab<0>(false, p, grid, pl.threads, st); break;
        case 1: launch_slab<1>(false, p, grid, pl.threads, st); break;
        case 2: launch_slab<2>(false, p, grid, pl.threads, st); break;
        case 4: launch_slab<4>(false, p, grid, pl.threads, st); break;
        default: launch_slab<8>(false, p, grid, pl.threads, st); break;
    }
    return 0;
}

}  // namespace ub
