// igemm_rows_kernel -- persistent tcgen05 implicit GEMM for 3x3 / 1x1 convolution fprop and dgrad on NHWC bf16 images
// whose width divides 256 (W = 16, 32, 64, 128): the kernel of the 64x64 / 32x32 / 16x16 levels of the U-Net.
//
// Why a second main loop: igemm_conv_kernel fetches a 128-pixel activation box AND a weight tile for every (tap,
// 64-channel block), one CTA per 128 pixels; at C = 64..192 that is 3.4 KB of L2->SMEM traffic per output pixel and a
// prologue + pipeline fill + epilogue per 128 pixels, and the layers ran at 15-25 % of the tensor peak.  Here
//   * a tile is TH = 256 / W whole image rows (M = 256 = two UMMA M=128 halves sharing every weight tile);
//   * the activations of a 64-channel block are loaded as THREE boxes (dx = -1, 0, +1), each (TH + 2) rows x W pixels
//     with TMA zero fill as the padding; the three dy taps of a box are descriptor start offsets of dy * W * 128 B --
//     multiples of 1024 B, so every MMA reads 1024-byte-aligned swizzle atoms (the first halo experiment derived all 9
//     taps from one box, and its 128-byte-shifted starts doubled the MMA time: profiles/r01_ncu_halo_*);
//   * the CTA is persistent (one per SM, static round-robin over tiles): TMEM holds two accumulator sets, so the
//     epilogue of tile i (8 warps: TMEM lane quadrant x M half) overlaps the main loop of tile i+1, and barrier init /
//     TMEM allocation / descriptor prefetch are paid once per SM instead of once per 128 pixels.
//
//   A ring : boxes (64 ch, W, TH+2, 1) of (TH+2)*W*128 B (36-48 KiB), 2-4 stages
//   W ring : (tap, 64-ch block) weight tiles BN x 64, 2-8 stages, order (block, dx, dy) to match the A boxes
//   TMEM   : 2 tile buffers x 2 halves x BN fp32 columns (BN <= 128)
//   warps  : 0 = A producer, 1 = W producer, 2 = MMA issuer of M half 0 + TMEM allocator, 3 = MMA issuer of M half 1,
//            4-11 = epilogue
// Same epilogue (bias / embedding vector / residual / GroupNorm hooks) as igemm_conv_kernel: epilogue.cuh.
#include "epilogue.cuh"
#include "igemm.cuh"
#include "launch.cuh"
#include "ptx.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#ifdef UB_TRACE
#include <algorithm>
#include <vector>
#endif

namespace ub {

static constexpr int kRowsThreads = 384;
static constexpr int kRowsEpiThreads = 256;
static constexpr int kMaxAStages = 4;
static constexpr int kMaxWStages = 16;

// Phase timeline of igemm_rows_kernel (development only: -DUB_TRACE, build/igemm_trace shape ... halo=1).  Per CTA and
// per tile of its schedule: SM clock (relative to CTA entry) at
//   [0] A producer: first box issued  [1] last box issued  [2] W producer: last tile issued
//   [3] MMA warp: accumulator buffer free (t_empty)  [4] first A box landed  [5] last MMA issued
//   [6] epilogue: accumulator complete (t_full)  [7] epilogue done
#ifdef UB_TRACE
static constexpr int kRTiles = 6, kRSlots = 8, kRCtas = 160;
__device__ unsigned long long g_rows_trace[kRCtas * kRTiles * kRSlots];
__device__ unsigned long long g_rows_t0[kRCtas];
#define UB_RTR(tile_i, slot)                                                                               \
    do {                                                                                                   \
        if ((threadIdx.x & 31) == 0 && int(blockIdx.x) < kRCtas && (tile_i) < kRTiles)                     \
            g_rows_trace[(int(blockIdx.x) * kRTiles + (tile_i)) * kRSlots + (slot)] = clock64();            \
    } while (0)
void igemm_rows_trace_dump(int nctas, int ntiles_total) {
    std::vector<unsigned long long> h(size_t(kRCtas) * kRTiles * kRSlots), t0(kRCtas);
    cudaMemcpyFromSymbol(h.data(), g_rows_trace, h.size() * 8);
    cudaMemcpyFromSymbol(t0.data(), g_rows_t0, t0.size() * 8);
    nctas = std::min(nctas, kRCtas);
    const char* names[kRSlots] = {"A first box issued", "A last box issued", "W last tile issued", "MMA: tmem buffer free",
                                  "MMA: first A landed", "MMA: last MMA issued", "EPI: accumulator ready", "EPI: done"};
    for (int t = 0; t < kRTiles; ++t) {
        int n = 0;
        double sum[kRSlots] = {0};
        for (int c = 0; c < nctas; ++c) {
            if (c + t * nctas >= ntiles_total) continue;
            ++n;
            for (int k = 0; k < kRSlots; ++k) sum[k] += double(h[(size_t(c) * kRTiles + t) * kRSlots + k] - t0[c]);
        }
        if (!n) break;
        printf("  rows trace, tile #%d of the CTA (%d CTAs):", t, n);
        for (int k = 0; k < kRSlots; ++k) printf("  %s %.0f", names[k], sum[k] / n);
        printf("\n");
    }
}
#else
#define UB_RTR(tile_i, slot) do {} while (0)
#endif

struct RowsBars {
    uint64_t a_full[kMaxAStages], a_empty[kMaxAStages];
    uint64_t w_full[kMaxWStages], w_empty[kMaxWStages];
    uint64_t t_full[2], t_empty[2];
    uint32_t tmem_slot;
    uint32_t pad_[3];
};
// smem tail behind the rings (floats): comb[2][BN] | gconst[2][4][BN] | red[8][BN][2]
// (16 epilogue warps -- a column split on top of quadrant x half -- measured 20 % slower: the 102-register cap of a
// 640-thread CTA spills in the hooked chunk)
static size_t rows_tail_floats(int BN) { return size_t(2 + 8 + 16) * BN; }

__global__ void __launch_bounds__(kRowsThreads, 1) igemm_rows_kernel(const __grid_constant__ IgemmRowsParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;
    uint8_t* sW = smem + size_t(p.a_stages) * p.a_stage_bytes;
    RowsBars* bars = reinterpret_cast<RowsBars*>(sW + size_t(p.w_stages) * p.w_stage_bytes);
    float* comb = reinterpret_cast<float*>(bars + 1);
    float* gconst = comb + 2 * p.BN;
    float* red = gconst + 8 * p.BN;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_mb = p.B * p.tiles_per_img;  // pixel tiles; the N tile is the slow index of the schedule
#ifdef UB_TRACE
    if (threadIdx.x == 0 && int(blockIdx.x) < kRCtas) g_rows_t0[blockIdx.x] = clock64();
#endif

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.nseg; ++s) {
            tma_prefetch_desc(&p.seg[s].tmA);
            tma_prefetch_desc(&p.seg[s].tmW);
        }
        // (two MMA issuers -- one per M half -- release every stage and complete every accumulator set together)
        for (int i = 0; i < p.a_stages; ++i) mbar_init(&bars->a_full[i], 1), mbar_init(&bars->a_empty[i], 2);
        for (int i = 0; i < p.w_stages; ++i) mbar_init(&bars->w_full[i], 1), mbar_init(&bars->w_empty[i], 2);
        for (int i = 0; i < 2; ++i) mbar_init(&bars->t_full[i], 2), mbar_init(&bars->t_empty[i], 8);
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc(&bars->tmem_slot, 512);
        tmem_relinquish();
    }
    if (warp == 4 && lane == 0 && p.epi.gn_x && int(blockIdx.x) < p.num_tiles) {  // first tile's GN-input rows -> L2
        const int mt = int(blockIdx.x) % tiles_mb;
        const int b = mt / p.tiles_per_img, h0 = (mt % p.tiles_per_img) * p.TH;
        l2_prefetch_bulk(p.epi.gn_x + ((size_t(b) * p.H + h0) * p.W) * p.epi.gn_ldx,
                         (uint32_t(min(p.TH, p.H - h0) * p.W - 1) * uint32_t(p.epi.gn_ldx) + uint32_t(p.Cout)) * 2u);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_slot;
    pdl_wait();  // everything above touched only kernel parameters, shared memory and TMEM

    if (warp == 0) {
        // ------------------------------------------------------------------ A producer: one box per (block, dx)
        // (whole warp converged, instructions under elect.sync: see elect_one_sync in ptx.cuh)
        {
            int st = 0;
            uint32_t ph = 0;
            int ti = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++ti) {
                const int mt = tile % tiles_mb;
                const int b = mt / p.tiles_per_img, h0 = (mt % p.tiles_per_img) * p.TH;
                for (int s = 0; s < p.nseg; ++s) {
                    const int ndx = p.seg[s].ntaps == 9 ? 3 : 1;
                    for (int cb = 0; cb < p.seg[s].cblocks; ++cb)
                        for (int dxi = 0; dxi < ndx; ++dxi) {
                            mbar_wait(&bars->a_empty[st], ph ^ 1);
                            if (s == 0 && cb == 0 && dxi == 0) UB_RTR(ti, 0);
                            UB_RTR(ti, 1);
                            if (elect_one_sync()) {
                                mbar_expect_tx(&bars->a_full[st], p.a_bytes);
                                tma_load_4d(sA + size_t(st) * p.a_stage_bytes, &p.seg[s].tmA, &bars->a_full[st], cb * 64,
                                            ndx == 3 ? dxi - 1 : 0, ndx == 3 ? h0 - 1 : h0, b);
                            }
                            __syncwarp();
                            if (++st == p.a_stages) st = 0, ph ^= 1;
                        }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ W producer: (block, dx, dy) order
        {
            int st = 0;
            uint32_t ph = 0;
            int ti = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++ti) {
                if (p.w_resident && ti > 0) break;  // resident weights: the ring was filled for the first tile, for good
                const int n0 = (tile / tiles_mb) * p.BN;
                for (int s = 0; s < p.nseg; ++s) {
                    const int nd = p.seg[s].ntaps == 9 ? 3 : 1;
                    for (int cb = 0; cb < p.seg[s].cblocks; ++cb)
                        for (int dxi = 0; dxi < nd; ++dxi)
                            for (int dyi = 0; dyi < nd; ++dyi) {
                                const int tap = dyi * 3 + dxi;  // (0 for a 1x1 segment)
                                mbar_wait(&bars->w_empty[st], ph ^ 1);
                                UB_RTR(ti, 2);
                                if (elect_one_sync()) {
                                    mbar_expect_tx(&bars->w_full[st], p.w_bytes);
                                    tma_load_2d(sW + size_t(st) * p.w_stage_bytes, &p.seg[s].tmW, &bars->w_full[st],
                                                cb * 64, tap * p.Cout + n0);
                                }
                                __syncwarp();
                                if (++st == p.w_stages) st = 0, ph ^= 1;
                            }
                }
            }
        }
    } else if (warp == 2 || warp == 3) {
        // ------------------------------------------------------------------ MMA issuers: warp 2 -> M half 0, warp 3 -> 1
        // (whole warp converged, MMAs / commits under elect.sync: see elect_one_sync in ptx.cuh)
        {
            const int mhalf = warp - 2;
            const uint32_t idesc = make_idesc_bf16(128, p.BN, 0, 0);
            const uint32_t row_bytes = uint32_t(p.W) * 128u;  // one image row of a box (multiple of 1024)
            int sa = 0, sw = 0;
            uint32_t pa = 0, pw = 0;
            int it = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
                const int buf = it & 1;
                mbar_wait(&bars->t_empty[buf], ((it >> 1) & 1) ^ 1);
                if (mhalf == 0) UB_RTR(it, 3);
                tc_fence_after();
                const uint32_t d0 = tmem_base + uint32_t(buf * 2 * p.BN);
                bool first = true;
                for (int s = 0; s < p.nseg; ++s) {
                    const int nd = p.seg[s].ntaps == 9 ? 3 : 1;
                    for (int cb = 0; cb < p.seg[s].cblocks; ++cb)
                        for (int dxi = 0; dxi < nd; ++dxi) {
                            mbar_wait(&bars->a_full[sa], pa);
                            if (mhalf == 0 && first) UB_RTR(it, 4);
                            tc_fence_after();
                            const uint32_t a_base = smem_u32(sA + size_t(sa) * p.a_stage_bytes);
                            for (int dyi = 0; dyi < nd; ++dyi) {
                                if (!p.w_resident || it == 0) mbar_wait(&bars->w_full[sw], pw);
                                tc_fence_after();
                                const uint32_t a0 = a_base + uint32_t(dyi) * row_bytes;  // box starts at row h0 - 1
                                const uint64_t dB =
                                    make_smem_desc_sw128(smem_u32(sW + size_t(sw) * p.w_stage_bytes), 16, 1024);
                                const uint64_t dA = make_smem_desc_sw128(a0 + uint32_t(mhalf) * 16384u, 16, 1024);
                                if (elect_one_sync()) {
#pragma unroll
                                    for (int k = 0; k < 4; ++k)
                                        umma_bf16(d0 + uint32_t(mhalf * p.BN), dA + uint64_t(k * 2), dB + uint64_t(k * 2),
                                                  idesc, (!first || k != 0) ? 1u : 0u);
                                    if (!p.w_resident) umma_commit(&bars->w_empty[sw]);
                                    if (dyi == nd - 1) umma_commit(&bars->a_empty[sa]);
                                }
                                __syncwarp();
                                first = false;
                                if (++sw == p.w_stages) sw = 0, pw ^= 1;
                            }
                            if (++sa == p.a_stages) sa = 0, pa ^= 1;
                        }
                }
                if (mhalf == 0) UB_RTR(it, 5);
                if (elect_one_sync()) umma_commit(&bars->t_full[buf]);
                __syncwarp();
            }
        }
    } else if (warp >= 4) {
        // ------------------------------------------------------------------ epilogue: quadrant q of M half `half`
        const int q = warp & 3, half = (warp - 4) >> 2;
        const int et = threadIdx.x - 128;
        EpiOut eo = epi_out(p.epi, p.Cout, p.H, p.W);
        const bool hook = p.epi.stats || p.epi.gn_x;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
            const int n0 = (tile / tiles_mb) * p.BN;
            const int mt = tile % tiles_mb;
            const int b = mt / p.tiles_per_img, h0 = (mt % p.tiles_per_img) * p.TH;
            const int buf = it & 1;
            // stage the per-channel addend (and the GroupNorm constants) of this tile while its MMAs are running;
            // double buffered: a fast warp may stage tile i+1 while a slow one still reads tile i's
            float* cb_ = comb + buf * p.BN;
            float* gc_ = gconst + buf * 4 * p.BN;
            epi_stage_comb(cb_, p.epi.bias, p.epi.bias2, p.epi.rowvec, b, p.Cout, n0, p.BN, et, kRowsEpiThreads);
            if (p.epi.gn_x)
                epi_stage_gconst(gc_, p.epi.gn_chsum, p.epi.gn_gamma, p.epi.gn_beta, b, p.Cout, p.epi.gn_cpg, p.H * p.W,
                                 n0, p.BN, et, kRowsEpiThreads);
            named_bar_sync(1, kRowsEpiThreads);
            if (p.epi.gn_x && threadIdx.x == 128) {
                // the NEXT tile's GroupNorm-input rows (written in the forward pass, long evicted) -> L2
                const int nt = tile + int(gridDim.x);
                if (nt < p.num_tiles) {
                    const int nmt = nt % tiles_mb;
                    const int nb = nmt / p.tiles_per_img, nh0 = (nmt % p.tiles_per_img) * p.TH;
                    const int nrows = min(p.TH, p.H - nh0);
                    l2_prefetch_bulk(p.epi.gn_x + ((size_t(nb) * p.H + nh0) * p.W) * p.epi.gn_ldx,
                                     (uint32_t(nrows * p.W - 1) * uint32_t(p.epi.gn_ldx) + uint32_t(p.Cout)) * 2u);
                }
            }
            const int row = half * 128 + q * 32 + lane;
            const int h = h0 + row / p.W, w = row % p.W;
            const bool valid = h < p.H;
            const size_t pix = (size_t(b) * p.H + h) * p.W + w;
            uint4 side[2];
            if (hook) epi_side_load(eo, valid, pix, n0, side);  // hidden behind the tile's main loop
            mbar_wait(&bars->t_full[buf], (it >> 1) & 1);
            if (warp == 4) UB_RTR(it, 6);
            if (tile + int(gridDim.x) >= p.num_tiles) pdl_trigger_late();  // last tile of this CTA
            tc_fence_after();
            const uint32_t trow = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(buf * 2 * p.BN + half * p.BN);
            epi_row(eo, trow, cb_, p.BN, valid, pix, b, h, w, n0, gc_, lane, red + size_t(warp - 4) * p.BN * 2, 0, 1,
                    side);
            // all TMEM reads of this buffer are complete (tcgen05.wait::ld above): hand it back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (warp == 4) UB_RTR(it, 7);
            if (lane == 0) mbar_arrive(&bars->t_empty[buf]);
            if (hook) {  // the 8 warps' column sums of this tile (one image) -> one vector RED per channel
                named_bar_sync(2, kRowsEpiThreads);
                float* dst = p.epi.gn_x ? p.epi.gn_S : p.epi.stats;
                for (int c = et; c < p.BN; c += kRowsEpiThreads) {
                    float s0 = 0.f, s1 = 0.f;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const float2 v = *reinterpret_cast<const float2*>(red + (size_t(k) * p.BN + c) * 2);
                        s0 += v.x, s1 += v.y;
                    }
                    float* d = dst + (size_t(b) * p.Cout + n0 + c) * 2;
                    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(d), "f"(s0), "f"(s1) : "memory");
                }
                // (the next tile's writes to `red` come after its named_bar_sync(1), i.e. after every thread is here)
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------ host
bool igemm_rows_eligible(int B, int H, int W, int Cout) {
    (void)B;
    if (W < 16 || W > 128 || (256 % W) != 0) return false;
    if (H < 256 / W) return false;  // a tile is 256 / W rows of ONE image
    if (Cout % 16 != 0) return false;
    return true;
}

int igemm_rows_plan(IgemmRowsParams* p, const ConvSegDesc* segs, int nseg, int B, int H, int W, int Cout,
                    const ConvEpilogue& ep, int sm_count) {
    memset(p, 0, sizeof(*p));
    if (nseg < 1 || nseg > 2 || !igemm_rows_eligible(B, H, W, Cout)) return -1;
    const bool gn_hook = ep.stats || ep.gn_x;
    int BN = 0;
    for (int cand = 128; cand >= 16; cand -= 16)
        if (Cout % cand == 0 && (!gn_hook || cand % 32 == 0)) {
            BN = cand;
            break;
        }
    if (!BN) return -2;
    p->nseg = nseg, p->B = B, p->H = H, p->W = W, p->Cout = Cout, p->BN = BN;
    p->TH = 256 / W;
    p->tiles_per_img = (H + p->TH - 1) / p->TH;
    p->num_tiles = B * p->tiles_per_img * (Cout / BN);
    int ntaps0 = segs[0].ntaps;
    for (int s = 0; s < nseg; ++s)
        if (segs[s].ntaps == 9) ntaps0 = 9;
    // every segment uses the same box shape: (TH + 2) rows when any segment is 3x3 -- a 1x1 segment then loads its box
    // from row h0 and leaves the last two rows unused
    const int box_rows = ntaps0 == 9 ? p->TH + 2 : p->TH;
    p->box_rows = box_rows;
    p->a_bytes = uint32_t(64 * W * box_rows * 2);
    p->a_stage_bytes = (p->a_bytes + 1023u) & ~1023u;
    p->w_bytes = uint32_t(64 * BN * 2);
    p->w_stage_bytes = (p->w_bytes + 1023u) & ~1023u;
    const size_t fixed = 1024 + sizeof(RowsBars) + rows_tail_floats(BN) * sizeof(float);
    const size_t budget = size_t(227) * 1024 - fixed;
    int as = 3, ws = 0;
    for (; as >= 2; --as) {
        if (size_t(as) * p->a_stage_bytes >= budget) continue;
        ws = int((budget - size_t(as) * p->a_stage_bytes) / p->w_stage_bytes);
        if (ws >= 3 || (as == 2 && ws >= 2)) break;
    }
    if (as < 2 || ws < 2) return -3;
    if (ws > kMaxWStages) ws = kMaxWStages;
    // The weight ring must cover the TMA round trip (~1300 cycles L2 hit + transfer, profiles/r02b_rows_trace.txt): with 4
    // stages of 8 KiB the W producer paced the 64-channel layers at ~700 cycles per (dx, dy) step against 384 cycles of
    // MMA work.  Spare room beyond 8 weight stages goes to a 4th A stage.
    if (as == 3 && ws > 8 && size_t(4) * p->a_stage_bytes + size_t(8) * p->w_stage_bytes <= budget) {
        as = 4;
        ws = int((budget - size_t(4) * p->a_stage_bytes) / p->w_stage_bytes);
        if (ws > kMaxWStages) ws = kMaxWStages;
    }
    // Resident weights: a layer whose whole weight set is one ring's worth -- a single segment of <= 64 input channels and
    // one N tile (the 64 -> 64 convs of the 64x64 level) -- loads its ntaps tiles ONCE per CTA; the ring has exactly ntaps
    // stages, the MMA issuers wait for them during their first tile only and never release them.  The 72 KiB of weight
    // traffic per 256-pixel tile (a third of the tile's bytes, nine barrier round trips) disappear.
    p->w_resident = 0;
    if (nseg == 1 && segs[0].Cin <= 64 && Cout == BN && ws >= segs[0].ntaps) {
        p->w_resident = 1;
        ws = segs[0].ntaps;
        // the room the shorter ring frees goes to the activation ring
        const int as2 = int((budget - size_t(ws) * p->w_stage_bytes) / p->a_stage_bytes);
        if (as2 > as) as = as2 > kMaxAStages ? kMaxAStages : as2;
    }
    p->a_stages = as, p->w_stages = ws;
    for (int s = 0; s < nseg; ++s) {
        const ConvSegDesc& d = segs[s];
        if ((d.ntaps != 9 && d.ntaps != 1) || d.Cin % 8 != 0) return -4;
        int r = make_act_map(&p->seg[s].tmA, d.x, d.Cin, d.ldx, W, H, B, W, box_rows, 1);
        if (r) return r;
        r = make_bf16_map_2d(&p->seg[s].tmW, d.wp, d.Cin, d.ntaps * Cout, d.Cin, BN);
        if (r) return r;
        p->seg[s].cblocks = (d.Cin + 63) / 64;
        p->seg[s].ntaps = d.ntaps;
    }
    const int r = igemm_epi_plan(&p->epi, ep, Cout);
    if (r) return r;
    p->grid = p->num_tiles < sm_count ? p->num_tiles : sm_count;
    return 0;
}

void igemm_rows_init() {
    static bool done = false;
    if (done) return;
    cudaFuncSetAttribute(igemm_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(227 * 1024));
    done = true;
}

int igemm_rows_launch(const IgemmRowsParams& p, cudaStream_t st) {
    igemm_rows_init();
    const size_t smem = size_t(p.a_stages) * p.a_stage_bytes + size_t(p.w_stages) * p.w_stage_bytes + sizeof(RowsBars) +
                        rows_tail_floats(p.BN) * sizeof(float) + 1024;
    const cudaError_t e = launch_pdl(igemm_rows_kernel, dim3(p.grid), dim3(kRowsThreads), smem, st, p);
    if (e != cudaSuccess)
        fprintf(stderr, "[unet_b200] igemm_rows launch failed: %s (grid %d, smem %zu, BN %d, stages %d/%d)\n",
                cudaGetErrorString(e), p.grid, smem, p.BN, p.a_stages, p.w_stages);
    return int(e);
}

}  // namespace ub
