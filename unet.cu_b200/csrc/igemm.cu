// tcgen05 implicit-GEMM kernels for sm_100a: convolution fprop/dgrad and wgrad on NHWC bf16 operands.
//
// Both kernels are warp-specialised:
//   warp 0   : TMA producer (one elected lane) - stages halo-shifted activation boxes + weight boxes in smem
//   warp 1   : tcgen05.mma issuer (one elected lane) + TMEM allocator
//   conv     : warps 2-9 epilogue (two per TMEM lane quadrant) - tcgen05.ld accumulators out of TMEM, fuse bias / emb /
//              residual / GroupNorm hooks, store; in igemm_conv2/4_kernel lane 0 of the last epilogue warp(s) first
//              issues the extra MMA streams
//   wgrad    : warps 2-5 epilogue - TMA reduce-add boxes (staged in the idle operand ring) into the fp32 weight-gradient
//              buffers (two-pass mode of the layer API: plain stores of split-K partials)
// smem stages are handed over with mbarriers (full: TMA complete_tx, empty: tcgen05.commit).
//
// Reference behaviour being replaced (not its structure): /root/reference/dev/conv2d_k3.cu:679-740 (forward3),
// :1132-1174 (dx_backward), :2468-2547 (dweight_dbias_backward1), :1365-1393 (dweight_reduce_kernel).
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

static constexpr int kMaxStages = 8;
static constexpr int kConvThreads = 320;   // conv: TMA warp, MMA warp, 8 epilogue warps (2 per TMEM lane quadrant)
static constexpr int kWgradThreads = 192;  // wgrad: TMA warp, MMA warp, 4 epilogue warps
static constexpr int kEpiThreads = kConvThreads - 64;

// Phase timeline of igemm_conv_kernel (development only: -DUB_TRACE, tools/igemm_test.cu `trace` mode).  Per CTA:
// [0] globaltimer at entry, [1] SM id, then SM clock at [2] entry [3] prologue done [4] griddepcontrol.wait passed
// [5] last TMA issued [6] first stage landed [7] last MMA issued [8] accumulator complete [9] epilogue done [10] exit
// [11] globaltimer at exit.
#ifdef UB_TRACE
static constexpr int kTraceSlots = 12, kTraceCtas = 2048;
__device__ unsigned long long g_conv_trace[kTraceSlots * kTraceCtas];
// 0 = normal, 1 = TMA stream only (no MMAs: stages are released by a plain arrive), 2 = MMA stream only (no TMA, no
// full-barrier waits: the MMAs read whatever is in shared memory) -- which side paces the main loop?
__device__ int g_conv_dbg_mode;
void igemm_trace_set_mode(int m) { cudaMemcpyToSymbol(g_conv_dbg_mode, &m, sizeof(int)); }
__device__ __forceinline__ unsigned long long trace_gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define UB_TR(slot, val)                                                                              \
    do {                                                                                              \
        const unsigned cta_ = blockIdx.y * gridDim.x + blockIdx.x;                                    \
        if (cta_ < unsigned(kTraceCtas)) g_conv_trace[cta_ * kTraceSlots + (slot)] = (val);           \
    } while (0)
void igemm_trace_dump(int nctas, double clock_ghz) {
    std::vector<unsigned long long> h(size_t(kTraceSlots) * kTraceCtas);
    cudaMemcpyFromSymbol(h.data(), g_conv_trace, h.size() * sizeof(unsigned long long));
    if (nctas > kTraceCtas) nctas = kTraceCtas;
    unsigned long long g0 = ~0ull, g1 = 0, gs_max = 0;
    for (int i = 0; i < nctas; ++i) {
        g0 = std::min(g0, h[size_t(i) * kTraceSlots]);
        gs_max = std::max(gs_max, h[size_t(i) * kTraceSlots]);
        g1 = std::max(g1, h[size_t(i) * kTraceSlots + 11]);
    }
    const char* names[] = {"prologue(sync)", "pdl_wait", "last TMA issued", "first stage landed", "last MMA issued",
                           "accumulator complete", "epilogue done", "exit"};
    printf("  trace: %d CTAs, first entry -> last exit %.2f us, entry spread %.2f us\n", nctas, (g1 - g0) * 1e-3,
           (gs_max - g0) * 1e-3);
    for (int k = 3; k <= 10; ++k) {
        double sum = 0, mx = 0, mn = 1e30;
        for (int i = 0; i < nctas; ++i) {
            const double d = double(h[size_t(i) * kTraceSlots + k] - h[size_t(i) * kTraceSlots + 2]);
            sum += d, mx = std::max(mx, d), mn = std::min(mn, d);
        }
        printf("    %-22s  avg %8.0f clk (%6.2f us)  min %8.0f  max %8.0f\n", names[k - 3], sum / nctas,
               sum / nctas / (clock_ghz * 1e3), mn, mx);
    }
}
#else
#define UB_TR(slot, val) do {} while (0)
#endif

// =====================================================================================================
// fprop / dgrad / 1x1 / linear
// =====================================================================================================
// One K block (stage) worth of MMAs for issuer `issuer` of NACC: K blocks it = issuer (mod NACC), accumulator `issuer`.
template <int NACC>
__device__ __forceinline__ void conv_issue_loop(const IgemmConvParams& p, int issuer, int nk, uint8_t* smem,
                                                uint64_t* full_bar, uint64_t* empty_bar, uint64_t* tmem_full_bar,
                                                uint32_t tmem_base) {
    const uint32_t idesc = make_idesc_bf16(128, p.BN, 0, 0);
    const uint32_t d = tmem_base + uint32_t(issuer * p.BN);
    // (NACC > 1: the ring is a multiple of NACC -- plan -- so stage s always belongs to issuer s % NACC and each
    //  issuer waits for consecutive phases of its full barriers)
    int stage = issuer;
    uint32_t phase = 0;
#ifdef UB_TRACE
    const int dbg = g_conv_dbg_mode;
#endif
    // The WHOLE warp runs this loop (converged); only the instruction block is under elect.sync -- see elect_one_sync.
    for (int it = issuer; it < nk; it += NACC) {
#ifdef UB_TRACE
        if (dbg < 2)
#endif
        mbar_wait(&full_bar[stage], phase);
        if (it == 0) UB_TR(6, (unsigned long long)clock64());
        tc_fence_after();
        const uint32_t sA = smem_u32(smem + size_t(stage) * p.stage_bytes);
        const uint32_t sB = sA + 16384;
        const uint64_t dA = make_smem_desc_sw128(sA, 16, 1024);
        const uint64_t dB = make_smem_desc_sw128(sB, 16, 1024);
#ifdef UB_TRACE
        if (dbg == 1) {
            if (elect_one_sync()) mbar_arrive(&empty_bar[stage]);
        } else
#endif
        if (elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                // advance 16 bf16 (32 B) along K inside the 128-byte swizzle row: +2 in the >>4 address field
                umma_bf16(d, dA + uint64_t(k * 2), dB + uint64_t(k * 2), idesc, (it >= NACC || k != 0) ? 1u : 0u);
            }
            umma_commit(&empty_bar[stage]);
        }
        __syncwarp();
        stage += NACC;
        if (stage >= p.stages) stage -= p.stages, phase ^= 1;
    }
#ifdef UB_TRACE
    if (dbg == 1) {
        if (elect_one_sync()) mbar_arrive(tmem_full_bar);
    } else
#endif
    if (elect_one_sync()) umma_commit(tmem_full_bar);
    __syncwarp();
    if (issuer == 0) UB_TR(7, (unsigned long long)clock64());
}

// TMA producer `prod` of NPROD: K blocks it = prod (mod NPROD) into stage it % stages (NPROD > 1: the ring is a
// multiple of NPROD, so a stage always belongs to the same producer).  One thread's TMA issue rate is part of what
// paces a one-CTA-per-SM pipeline: tools/tma_ingest_bench.cu NPROD=2 moves 68 B/clk/SM through one-box stages against
// 50 with a single producer warp (123 against 92 with two boxes per stage, profiles/r02_tma_producers.txt).
template <int NPROD>
__device__ __forceinline__ void conv_produce_loop(const IgemmConvParams& p, int prod, int /*nk*/, uint8_t* smem,
                                                  uint64_t* full_bar, uint64_t* empty_bar, int w0, int h0, int b0,
                                                  int n0) {
    // (nested loops over segment / tap / channel block with the K blocks of the other producers skipped: a flat loop
    //  that derives (segment, tap, block) per iteration cost 130 cycles more per K block in the phase trace)
    int stage = prod, it = 0;
    uint32_t phase = 0;
    for (int s = 0; s < p.nseg; ++s) {
        const IgemmSeg& sg = p.seg[s];
        for (int tap = 0; tap < sg.ntaps; ++tap) {
            const int dy = sg.ntaps == 9 ? tap / 3 - 1 : 0;
            const int dx = sg.ntaps == 9 ? tap % 3 - 1 : 0;
            for (int cb = 0; cb < sg.cblocks; ++cb, ++it) {
                if (NPROD > 1 && (it % NPROD) != prod) continue;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* sA = smem + size_t(stage) * p.stage_bytes;
                uint8_t* sB = sA + 16384;
                if (elect_one_sync()) {
                    mbar_expect_tx(&full_bar[stage], p.a_bytes + p.b_bytes);
                    tma_load_4d(sA, &sg.tmA, &full_bar[stage], cb * 64, w0 + dx, h0 + dy, b0);
                    tma_load_2d(sB, &sg.tmW, &full_bar[stage], cb * 64, tap * p.Cout + n0);
                }
                __syncwarp();
                stage += NPROD;
                if (stage >= p.stages) stage -= p.stages, phase ^= 1;
            }
        }
    }
}

// NACC = number of MMA issue streams (and accumulators).  One thread's tcgen05.mma stream runs at ~145 cycles per
// M=128 instruction whatever N is, and streams of different warps / CTAs overlap (profiles/r01_mma_issue.txt).  Grids
// that fill the chip run NACC = 1 with two CTAs per SM (two streams per SM already).  Grids of <= one CTA per SM (the
// 8x8 / 16x16 levels) run NACC = 2: lane 0 of the last epilogue warp -- idle during the main loop -- issues the odd K
// blocks into a second accumulator and the epilogue adds the two.  (An 11th warp for the second issuer capped the
// two-CTA kernel at 80 registers; the spilling epilogue cost more in the step than the main loop won.)
template <int NACC, bool MS = false>
__device__ __forceinline__ void igemm_conv_body(const IgemmConvParams& p) {
#ifdef UB_TRACE
    if (threadIdx.x == 0) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        UB_TR(0, trace_gtime());
        UB_TR(1, smid);
        UB_TR(2, (unsigned long long)clock64());
    }
#endif
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + size_t(p.stages) * p.stage_bytes);
    uint64_t* empty_bar = full_bar + kMaxStages;
    uint64_t* tmem_full_bar = empty_bar + kMaxStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
    // [ncomb][BN] staged per-channel addend (one row per image of the tile), 16-byte aligned behind the barriers
    float* comb = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);
    float* gconst = comb + p.ncomb * p.BN;  // [ngimg][4][BN] GroupNorm constants (gn-bwd epilogue only)
    float* red = gconst + p.ngimg * 4 * p.BN;  // [4 warps][BN][2] column sums of the GroupNorm hooks

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    // tile coordinates
    int t = blockIdx.x;
    const int tw = t % p.tiles_w;
    t /= p.tiles_w;
    const int th = t % p.tiles_h;
    const int tb = t / p.tiles_h;
    const int w0 = tw * p.TW, h0 = th * p.TH, b0 = tb * p.TB;
    const int n0 = blockIdx.y * p.BN;

    int nk = 0;
    for (int s = 0; s < p.nseg; ++s) nk += p.seg[s].ntaps * p.seg[s].cblocks;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < p.nseg; ++s) {
            tma_prefetch_desc(&p.seg[s].tmA);
            tma_prefetch_desc(&p.seg[s].tmW);
        }
        for (int i = 0; i < p.stages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        mbar_init(tmem_full_bar, NACC);
        if constexpr (MS) mbar_init(tmem_full_bar + 2, 1);  // statistics MMAs complete (byte 144 of the barrier block)
        fence_mbar_init();
    }
    if (warp == 1) {
        tmem_alloc(tmem_slot, p.tmem_cols);
        tmem_relinquish();
    }
    if (warp == 2 && lane == 0) {
        // Pull this N tile's weights into L2 while the previous kernel is still in its epilogue (late PDL trigger):
        // the weights are evicted by the ~2 GB of activations every step streams through the 126 MB L2, and the
        // low-resolution layers are paced by their weight tiles' latency.  The tile's rows of one tap are contiguous;
        // the pixel tiles of the grid share the taps.  (Packed weights are written by the optimizer's re-pack long
        // before -- never by the kernel this launch depends on.)
        for (int s = 0; s < p.nseg; ++s)
            for (int tap = blockIdx.x; tap < p.seg[s].ntaps; tap += gridDim.x)
                l2_prefetch_bulk(p.seg[s].wp + (size_t(tap) * p.Cout + n0) * p.seg[s].Cin,
                                 uint32_t(p.BN) * uint32_t(p.seg[s].Cin) * 2u);
    }
    if (warp == 3 && lane == 0 && p.epi.gn_x) {
        // gn-bwd hook: the GroupNorm input rows of this pixel tile were written in the forward pass (long evicted);
        // fetch them into L2 now instead of at the epilogue's dependent per-chunk loads.  A pixel row of the tile is
        // contiguous over all channels; the N tiles of the grid share the rows.
        const int nrows = p.TB * p.TH;
        for (int r = blockIdx.y; r < nrows; r += gridDim.y) {
            const int b = b0 + r / p.TH, h = h0 + r % p.TH;
            if (b < p.B && h < p.H) {
                const int wn = min(p.TW, p.W - w0);
                l2_prefetch_bulk(p.epi.gn_x + ((size_t(b) * p.H + h) * p.W + w0) * p.epi.gn_ldx,
                                 (uint32_t(wn - 1) * uint32_t(p.epi.gn_ldx) + uint32_t(p.Cout)) * 2u);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) UB_TR(3, (unsigned long long)clock64());
    pdl_wait();  // everything above touched only kernel parameters, shared memory, TMEM (and prefetched weights)
    if (threadIdx.x == 0) UB_TR(4, (unsigned long long)clock64());

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer
        // (whole warp converged; the TMA instructions are issued under elect.sync -- see elect_one_sync)
#ifdef UB_TRACE
        if (g_conv_dbg_mode < 2) {
#else
        {
#endif
            // two-stream kernels (one CTA per SM): a second producer (warp 8, see below) takes the odd K blocks
            conv_produce_loop<NACC>(p, 0, nk, smem, full_bar, empty_bar, w0, h0, b0, n0);
            UB_TR(5, (unsigned long long)clock64());
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (stream 0)
        conv_issue_loop<NACC>(p, 0, nk, smem, full_bar, empty_bar, tmem_full_bar, tmem_base);
    } else {
        // ------------------------------------------------------------ epilogue (warps 2..9)
        if constexpr (NACC == 2) {  // second MMA stream first; the warp reconverges before it touches the epilogue
            if (warp == 9) conv_issue_loop<NACC>(p, 1, nk, smem, full_bar, empty_bar, tmem_full_bar, tmem_base);
            // ... and the second TMA producer (odd K blocks) on another epilogue warp that idles during the main loop
            if (warp == 8) {
#ifdef UB_TRACE
                if (g_conv_dbg_mode < 2)
#endif
                conv_produce_loop<2>(p, 1, nk, smem, full_bar, empty_bar, w0, h0, b0, n0);
            }
        }
        const int q = warp & 3;  // TMEM lane quadrant this warp may access
        const int half = (warp - 2) >> 2;  // the two warps of a quadrant split the columns
        const int row = q * 32 + lane;
        const int lw = row % p.TW;
        const int lh = (row / p.TW) % p.TH;
        const int lb = row / (p.TW * p.TH);
        const int w = w0 + lw, h = h0 + lh, b = b0 + lb;
        const bool valid = (lb < p.TB) && (w < p.W) && (h < p.H) && (b < p.B);
        // stage bias + bias2 + embedding vector while the main loop runs: one row per image of the tile when the
        // embedding vector is used (p.ncomb == TB), a single shared row otherwise
        const int et = threadIdx.x - 64;
        for (int i = 0; i < p.ncomb; ++i)
            epi_stage_comb(comb + i * p.BN, p.epi.bias, p.epi.bias2, p.epi.rowvec, min(b0 + i, p.B - 1), p.Cout, n0,
                           p.BN, et, kEpiThreads);
        for (int i = 0; i < p.ngimg; ++i)
            epi_stage_gconst(gconst + i * 4 * p.BN, p.epi.gn_chsum, p.epi.gn_gamma, p.epi.gn_beta, min(b0 + i, p.B - 1),
                             p.Cout, p.epi.gn_cpg, p.H * p.W, n0, p.BN, et, kEpiThreads);
        named_bar_sync(1, kEpiThreads);

        const size_t pix = (size_t(b) * p.H + h) * p.W + w;
        EpiOut eo = epi_out(p.epi, p.Cout, p.H, p.W);
        eo.nacc = NACC, eo.acc_stride = uint32_t(p.BN);
        uint4 side[2];
        // (the first side-input chunk of a hook is loaded here, hidden behind the main loop)
        if (p.epi.stats || p.epi.gn_x) epi_side_load(eo, valid, pix, n0 + 16 * half, side);

        mbar_wait(tmem_full_bar, 0);
        pdl_trigger_late();  // main loop complete: the next kernel's prologue may overlap this epilogue
        if (threadIdx.x == 64) UB_TR(8, (unsigned long long)clock64());
        tc_fence_after();

        bool done_ms = false;
        if constexpr (MS) {
            if (p.ms) {
                done_ms = true;
                // ---- statistics on the tensor core (see IgemmConvParams::ms).  The pipeline stages are dead.
                // ms == 2: no statistics, only the staged tile + TMA store (plain convs: the per-thread 16-byte stores
                // of a pixel-per-thread epilogue hit 32 different lines per instruction -- 8.6 B/clk/SM measured on the
                // 1x1 skip-conv dgrads of the 64x64 level, whose epilogue is all they do)
                const bool stat = p.ms == 1;
                uint64_t* stat_bar = tmem_full_bar + 2;
                const int atoms = p.BN / 64;
                const uint32_t ys = smem_u32(smem);
                const uint32_t ones_s = ys + uint32_t(atoms) * 16384u;
                if (stat)
                    for (int i = et; i < 1024; i += kEpiThreads)  // 128 pixel rows x 128 B of bf16 1.0
                        sts_v4_b32(ones_s + 16u * i, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
                const float* cmb = comb + (p.ncomb > 1 ? min(lb, p.ncomb - 1) : 0) * p.BN;
                const uint32_t rowoff = uint32_t(row >> 3) * 1024u + uint32_t(row & 7) * 128u;
                for (int c0 = 16 * half; c0 < p.BN; c0 += 32) {
                    uint32_t v[16];
                    epi_tmem_load16(eo, tmem_base + (uint32_t(q * 32) << 16) + uint32_t(c0), v);
                    uint4 r[2];
                    if (p.epi.residual && valid) {
                        const uint4* rp = reinterpret_cast<const uint4*>(p.epi.residual + pix * p.epi.ldr + n0 + c0);
                        r[0] = rp[0], r[1] = rp[1];
                    }
                    tmem_ld_wait();
                    float f[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) f[j] = valid ? __uint_as_float(v[j]) + cmb[c0 + j] : 0.f;
                    if (p.epi.residual && valid) {
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            float t[8];
                            unpack_bf16x8(r[j], t);
#pragma unroll
                            for (int i = 0; i < 8; ++i) f[j * 8 + i] += t[i];
                        }
                    }
                    uint32_t py[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const __nv_bfloat162 h2 = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
                        py[i] = *reinterpret_cast<const uint32_t*>(&h2);
                    }
                    // MN-major SW128 atom: row = pixel (128 B = 64 channels), 16-byte chunk index XOR (row % 8)
                    const uint32_t abase = uint32_t(c0 >> 6) * 16384u + rowoff;
                    const uint32_t ch = uint32_t((c0 & 63) >> 3), sw = uint32_t(row & 7);
                    sts_v4_b32(ys + abase + ((ch ^ sw) << 4), py[0], py[1], py[2], py[3]);
                    sts_v4_b32(ys + abase + (((ch + 1) ^ sw) << 4), py[4], py[5], py[6], py[7]);
                }
                fence_proxy_async_smem();
                tc_fence_before();
                named_bar_sync(1, kEpiThreads);
                // [image][16 cols]: sum y, behind the accumulators and the Gram matrices (IgemmConvParams::ms)
                const uint32_t t_stat = tmem_base + uint32_t(max(NACC, p.TB) * p.BN);
                if (threadIdx.x == 64) {
                    tc_fence_after();
                    for (int a = 0; a < atoms; ++a) tma_store_4d(smem + size_t(a) * 16384, &p.tmO, n0 + a * 64, w0, h0, b0);
                    bulk_commit_group();
                  if (stat) {
                    // sum y = Y^T x ones (N = 16, column 0 used).  sum y*y = the diagonal of the Gram matrix Y^T Y (N =
                    // BN), written over the accumulator columns, which the loop above has read: products of two bf16
                    // values are exact in fp32, so every y*y enters the fp32 sum exactly.  (A staged Y*Y operand is
                    // rounded to bf16, 2^-9 relative per term, which GroupNorm's E[y^2] - mean^2 amplifies by
                    // (mean^2 + var) / var: the variance was off by 7e-3 for channels with a 4-sigma offset,
                    // tests/test_conv_fused_gpu.py on a B200.)
                    const uint32_t idesc = make_idesc_bf16(uint32_t(p.BN), 16, 1, 1);
                    const uint32_t gdesc = make_idesc_bf16(uint32_t(p.BN), uint32_t(p.BN), 1, 1);
                    const uint64_t dbase = make_smem_desc_sw128(0, 16384, 1024);  // LBO = 64-channel atom, SBO = 8 rows
                    const uint64_t dY = dbase | uint64_t((ys >> 4) & 0x3FFF), dO = dbase | uint64_t((ones_s >> 4) & 0x3FFF);
                    const int kpi = 8 / p.TB;  // K steps (16 pixels) per image of the tile
                    for (int img = 0; img < p.TB; ++img)
                        for (int k = 0; k < kpi; ++k) {
                            const uint64_t ko = uint64_t((img * kpi + k) * 128);  // 16 rows x 128 B, in 16-byte units
                            umma_bf16(t_stat + uint32_t(img * 32), dY + ko, dO + ko, idesc, k != 0);
                            umma_bf16(tmem_base + uint32_t(img * p.BN), dY + ko, dY + ko, gdesc, k != 0);
                        }
                    umma_commit(stat_bar);
                  }
                }
                if (stat) {
                mbar_wait(stat_bar, 0);
                tc_fence_after();
                if (half == 0) {
                    // M = 128: channel m in TMEM lane m.  M = 64: channel m in lane (m % 16) + 32 * (m / 16).  The sum
                    // of squares of channel m is column m of its row of the Gram matrix.
                    const int c_w = p.BN == 128 ? q * 32 : q * 16;  // first channel of this warp's lanes
                    const int chn = c_w + lane;
                    const bool cv = p.BN == 128 || lane < 16;
                    const uint32_t lrow = uint32_t(q * 32) << 16;
                    for (int img = 0; img < p.TB; ++img) {
                        uint32_t sv[16], gv[32];
                        tmem_ld16(t_stat + lrow + uint32_t(img * 32), sv);
                        tmem_ld32(tmem_base + lrow + uint32_t(img * p.BN + c_w), gv);
                        tmem_ld_wait();
                        float ss = 0.f;
#pragma unroll
                        for (int j = 0; j < 32; ++j) ss = j == lane ? __uint_as_float(gv[j]) : ss;
                        if (cv && b0 + img < p.B) {
                            float* d = p.epi.stats + (size_t(b0 + img) * p.Cout + n0 + chn) * 2;
                            asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(d), "f"(__uint_as_float(sv[0])),
                                         "f"(ss)
                                         : "memory");
                        }
                    }
                }
                }  // stat
                // the Y tile has left shared memory (waiting for the reads only -- wait_group.read -- measured the same:
                // profiles/r02n_wgrad_tma_red.txt)
                if (threadIdx.x == 64) bulk_wait_group0();
            }
        }
        if (!done_ms) {
        // GroupNorm hooks: all 32 pixels of a warp lie in one image of the tile (plan)
        const int lbw = min(lb, p.TB - 1);
        epi_row(eo, tmem_base + (uint32_t(q * 32) << 16), comb + (p.ncomb > 1 ? min(lb, p.ncomb - 1) : 0) * p.BN, p.BN,
                valid, pix, b, h, w, n0, gconst + lbw * 4 * p.BN, lane, red + size_t(q) * p.BN * 2, half, 2, side);
        if (p.epi.stats || p.epi.gn_x) {
            named_bar_sync(1, kEpiThreads);
            epi_flush_stats(red, p.epi.gn_x ? p.epi.gn_S : p.epi.stats, p.Cout, n0, p.BN, b0, p.B, p.TW * p.TH, p.TB,
                            et, kEpiThreads);
        }
        }  // !done_ms
        if (threadIdx.x == 64) UB_TR(9, (unsigned long long)clock64());
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, p.tmem_cols);
#ifdef UB_TRACE
    if (threadIdx.x == 0) {
        UB_TR(10, (unsigned long long)clock64());
        UB_TR(11, trace_gtime());
    }
#endif
}
__global__ void __launch_bounds__(kConvThreads, 2) igemm_conv_kernel(const __grid_constant__ IgemmConvParams p) {
    igemm_conv_body<1>(p);
}
__global__ void __launch_bounds__(kConvThreads, 1) igemm_conv2_kernel(const __grid_constant__ IgemmConvParams p) {
    igemm_conv_body<2>(p);
}
// tensor-core GroupNorm statistics + TMA output store, see IgemmConvParams::ms
__global__ void __launch_bounds__(kConvThreads, 2) igemm_conv_ms_kernel(const __grid_constant__ IgemmConvParams p) {
    igemm_conv_body<1, true>(p);
}
__global__ void __launch_bounds__(kConvThreads, 1) igemm_conv2_ms_kernel(const __grid_constant__ IgemmConvParams p) {
    igemm_conv_body<2, true>(p);
}

// =====================================================================================================
// wgrad: both operands MN-major (the contraction index is the pixel index, channels are contiguous)
// =====================================================================================================
__global__ void __launch_bounds__(kWgradThreads) igemm_wgrad_kernel(const __grid_constant__ IgemmWgradParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const uint32_t atom = uint32_t(p.KP) * 128u;  // one 64-channel operand atom: KP pixel rows of 128 B
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + size_t(p.stages) * p.stage_bytes + (p.ones_off ? atom : 0));
    uint64_t* empty_bar = full_bar + kMaxStages;
    uint64_t* tmem_full_bar = empty_bar + kMaxStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    const int n_ctiles = p.Cin / p.NC;
    const int o0 = (blockIdx.x / n_ctiles) * p.MO;
    const int c0 = (blockIdx.x % n_ctiles) * p.NC;
    const int tap0 = blockIdx.y * p.TC;
    const int split = blockIdx.z;

    const int ktiles = p.tiles_w * p.tiles_h * p.tiles_b;
    const int k_begin = int((long long)ktiles * split / p.nsplit);
    const int k_end = int((long long)ktiles * (split + 1) / p.nsplit);
    const int a_atoms = p.MO / 64, b_atoms = p.NC / 64;
    const uint32_t b_off = uint32_t(a_atoms) * atom;  // B region offset inside a stage
    // Column mode (3x3 layers, see IgemmWgradParams::colmode): blockIdx.y is the filter COLUMN dx + 1 and the CTA's
    // three taps are dy = -1, 0, +1 of that column, all read from ONE halo box of TH + 2 image rows per 64-channel atom.
    const bool colmode = p.colmode != 0;
    // fused bias gradient: only the CTAs that own the centre tap (or the single tap) of the first Cin tile
    // (row mode: filter row 1 holds taps 3..5; column mode: filter column 1 holds taps 1, 4, 7 -- blockIdx.y == 1 both)
    const int bias_ti = (p.ntaps == 9 ? 4 : 0) - tap0;
    const bool do_bias = p.ones_off != 0 && c0 == 0 && (colmode ? blockIdx.y == 1 : (bias_ti >= 0 && bias_ti < p.TC));
    if (do_bias) {  // KP pixel rows x 128 B of bf16 1.0 (any swizzle of a constant tile is the same tile)
        uint4* ones = reinterpret_cast<uint4*>(smem + p.ones_off);
        for (int i = threadIdx.x; i < p.KP * 8; i += blockDim.x) ones[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmDY);
        tma_prefetch_desc(&p.tmX);
        if (p.acc) tma_prefetch_desc(&p.tmAcc);
        for (int i = 0; i < p.stages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        mbar_init(tmem_full_bar, 1);
        fence_mbar_init();
    }
    if (warp == 1) {
        tmem_alloc(tmem_slot, p.tmem_cols);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();  // everything above touched only kernel parameters, shared memory and TMEM

    if (warp == 0) {
        // TMA producer (whole warp converged, TMA instructions under elect.sync: see elect_one_sync in ptx.cuh).
        // One producer: two lift single-box stages from ~52 to ~68 B/clk per SM (tools/tma_ingest_bench.cu), but these
        // stages hold 3-8 boxes and one producer already reaches ~72 -- a second producer warp measured no gain here
        // (measured, removed: profiles/r02n_wgrad_tma_red.txt).
        for (int kt = k_begin; kt < k_end; ++kt) {
            const int kl = kt - k_begin;
            const int stage = kl % p.stages;
            const uint32_t phase = uint32_t(kl / p.stages) & 1u;
            int t = kt;
            const int w0 = (t % p.tiles_w) * p.TW;
            t /= p.tiles_w;
            const int h0 = (t % p.tiles_h) * p.TH;
            const int b0 = (t / p.tiles_h) * p.TB;
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sA = smem + size_t(stage) * p.stage_bytes;
            uint8_t* sB = sA + b_off;
            if (elect_one_sync()) {
                mbar_expect_tx(&full_bar[stage], p.tx_bytes);
                // (the atom loops stay rolled: unrolled, they cost the kernel 700 instructions and 52 uniform-register
                //  spills to registers)
#pragma unroll 1
                for (int a = 0; a < a_atoms; ++a)
                    tma_load_4d(sA + a * atom, &p.tmDY, &full_bar[stage], o0 + a * 64, w0, h0, b0);
                if (colmode) {  // one (TH + 2)-row halo box per 64-channel atom, shifted by this CTA's dx
#pragma unroll 1
                    for (int nb = 0; nb < b_atoms; ++nb)
                        tma_load_4d(sB + nb * p.hatom, &p.tmX, &full_bar[stage], c0 + nb * 64,
                                    w0 + int(blockIdx.y) - 1, h0 - 1, b0);
                } else
                for (int ti = 0; ti < p.TC; ++ti) {
                    const int tap = tap0 + ti;
                    const int dy = p.ntaps == 9 ? tap / 3 - 1 : 0;
                    const int dx = p.ntaps == 9 ? tap % 3 - 1 : 0;
                    for (int nb = 0; nb < b_atoms; ++nb)
                        tma_load_4d(sB + (ti * b_atoms + nb) * atom, &p.tmX, &full_bar[stage], c0 + nb * 64, w0 + dx,
                                    h0 + dy, b0);
                }
            }
            __syncwarp();
        }
    }
    if (warp == 1) {
        {
            // Whole warp converged, MMAs / commits under elect.sync (see elect_one_sync in ptx.cuh).  Everything that does
            // not change per K tile is hoisted: descriptors are a constant high word plus the 16-byte-granular start
            // address, MMA groups are precomputed.
            const uint64_t dbase = make_smem_desc_sw128(0, atom, 1024);  // LBO = atom (64-channel atoms), SBO = 1024
            const int ksteps = p.KP / 16;
            const uint32_t idesc_b = make_idesc_bf16(p.MO, 16, 1, 1);
            const uint64_t d_ones = dbase | uint64_t((smem_u32(smem + p.ones_off) >> 4) & 0x3FFF);
            // taps are merged into MMAs of N <= 256: the B tiles of consecutive taps are consecutive 64-channel atoms
            // and their accumulators consecutive TMEM columns, so the dY operand is read once per group
            const int taps_per_mma = 256 / p.NC;
            int ng = 0;
            uint32_t g_col[3], g_boff[3], g_idesc[3];
            for (int ti = 0; ti < p.TC; ti += taps_per_mma, ++ng) {
                const int nt = min(taps_per_mma, p.TC - ti);
                g_col[ng] = uint32_t(ti * p.NC);
                g_boff[ng] = (b_off + uint32_t(ti * b_atoms) * atom) >> 4;
                g_idesc[ng] = make_idesc_bf16(p.MO, nt * p.NC, 1, 1);
            }
            // column mode: per 64-channel atom ONE N = 192 MMA per K step -- its three 64-channel N atoms are the three dy
            // windows of the halo box, TW pixels (one image row of the tile) apart: LBO = TW * 128 B, a multiple of the
            // 1 KiB swizzle atom, so every window starts aligned.  Accumulator columns: [atom][dy][64 channels].
            const uint64_t dbase_c = make_smem_desc_sw128(0, uint32_t(p.TW) * 128u, 1024);
            const uint32_t idesc_c = make_idesc_bf16(p.MO, 192, 1, 1);
            const uint32_t hatom16 = p.hatom >> 4, img_skip16 = uint32_t(p.TW) * 16u;  // (2 halo rows per image, in 16 B)
            const uint32_t s0 = smem_u32(smem);
            const uint32_t t_bias = tmem_base + uint32_t(p.TC * p.NC);
            int stage = 0;
            uint32_t phase = 0;
            for (int kt = k_begin; kt < k_end; ++kt) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                // 16 pixels (K) per MMA = 16 rows of 128 B = 2048 B = 128 descriptor units
                const uint64_t dA = dbase | uint64_t(((s0 + uint32_t(stage) * p.stage_bytes) >> 4) & 0x3FFF);
                const uint32_t acc0 = kt != k_begin;
                if (elect_one_sync()) {
                    if (do_bias) {
#pragma unroll 4
                        for (int k = 0; k < ksteps; ++k)
                            umma_bf16(t_bias, dA + uint64_t(k * 128), d_ones + uint64_t(k * 128), idesc_b,
                                      acc0 | uint32_t(k));
                    }
                    if (colmode) {
                        const uint64_t dB =
                            dbase_c | uint64_t(((s0 + uint32_t(stage) * p.stage_bytes + b_off) >> 4) & 0x3FFF);
                        for (int nb = 0; nb < b_atoms; ++nb) {
#pragma unroll 4
                            for (int k = 0; k < ksteps; ++k) {
                                // K step k = pixels [16 k, 16 k + 16) of the dY tile; in the halo box every image before
                                // it adds two rows
                                const uint32_t xo = uint32_t(k * 128) + (uint32_t(k * 16) >> p.lg_img) * img_skip16;
                                umma_bf16(tmem_base + uint32_t(nb * 192), dA + uint64_t(k * 128),
                                          dB + uint64_t(uint32_t(nb) * hatom16 + xo), idesc_c, acc0 | uint32_t(k));
                            }
                        }
                    } else {
#pragma unroll 3
                    for (int g = 0; g < ng; ++g) {
#pragma unroll 4
                        for (int k = 0; k < ksteps; ++k)
                            umma_bf16(tmem_base + g_col[g], dA + uint64_t(k * 128), dA + uint64_t(g_boff[g] + k * 128),
                                      g_idesc[g], acc0 | uint32_t(k));
                    }
                    }
                    umma_commit(&empty_bar[stage]);
                }
                __syncwarp();
                if (++stage == p.stages) {
                    stage = 0;
                    phase ^= 1;
                }
            }
            if (elect_one_sync()) umma_commit(tmem_full_bar);
            __syncwarp();
        }
    } else if (warp >= 2) {
        const int q = warp & 3;
        // M=128: accumulator row m lives in TMEM lane m.  M=64: row m lives in lane (m%16) + 32*(m/16).
        int row;
        bool valid;
        if (p.MO == 128) {
            row = q * 32 + lane;
            valid = true;
        } else {
            row = q * 16 + lane;
            valid = lane < 16;
        }
        mbar_wait(tmem_full_bar, 0);
        pdl_trigger_late();  // main loop complete: the next kernel's prologue may overlap this epilogue
        tc_fence_after();
        if (k_end > k_begin && p.acc) {
            // Accumulate mode through the TMA: thread = accumulator row, so a per-lane RED (or store) instruction touches
            // 32 different lines and the LSU takes one pass per lane -- 12 288 passes for a 128 x 384 tile, ~6 us, the
            // largest phase of the low-resolution launches (per-lane red.global.add: 1.31 ms per step for the weight
            // gradients against 1.19; measured, removed: profiles/r02n_wgrad_tma_red.txt).  Instead every warp stages
            // 32 columns of its MO/4 rows in the idle operand ring (fp32 rows of 128 B, 16-byte chunks XOR-swizzled
            // with the row: conflict-free STS.128 and the layout a SWIZZLE_128B box expects) and one elected lane
            // issues a reduce-add box per (tap, 32 columns); the L2 adds whole lines.  Warps are independent: each
            // owns a slice of the ring and re-uses a buffer only after its bulk group has read it.
            const int rpw = p.MO >> 2;  // accumulator rows of this warp: TMEM lanes 32q .. 32q + rpw - 1
            const uint32_t bufbytes = uint32_t(rpw) * 128u;
            const int nsub = p.NC >> 5, ntile = p.TC * nsub;
            int nbuf = int((uint32_t(p.stages) * p.stage_bytes / 4u) / bufbytes);
            if (nbuf > ntile) nbuf = ntile;
            const uint32_t wbase = smem_u32(smem) + uint32_t(q) * uint32_t(nbuf) * bufbytes;
            const uint32_t rowoff = uint32_t(lane) * 128u, sw = uint32_t(lane & 7);
            int slot = 0;
            for (int it = 0; it < ntile; ++it) {
                const int ti = it / nsub, s = it - ti * nsub;
                if (it != 0 && slot == 0) {  // wrapped around this warp's buffers
                    if (elect_one_sync()) bulk_wait_group_read0();
                    __syncwarp();
                }
                // accumulator column of (tap ti, channel s * 32): [ti][NC] in row mode, [atom][ti][64] in column mode
                const int tcol = colmode ? ((s >> 1) * 3 + ti) * 64 + (s & 1) * 32 : ti * p.NC + s * 32;
                uint32_t v[32];
                tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(tcol), v);
                tmem_ld_wait();
                const uint32_t buf = wbase + uint32_t(slot) * bufbytes;
                if (valid) {
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        sts_v4_b32(buf + rowoff + ((uint32_t(j) ^ sw) << 4), v[4 * j], v[4 * j + 1], v[4 * j + 2],
                                   v[4 * j + 3]);
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (elect_one_sync()) {
                    const int tap = colmode ? 3 * ti + int(blockIdx.y) : tap0 + ti;
                    tma_reduce_add_2d(buf, &p.tmAcc, c0 + s * 32, tap * p.Cout + o0 + q * rpw);
                    bulk_commit_group();
                }
                __syncwarp();
                if (++slot == nbuf) slot = 0;
            }
            if (elect_one_sync()) bulk_wait_group0();  // (the same lane committed every group: elect.sync is deterministic)
            __syncwarp();
        } else if (k_end > k_begin) {  // two-pass mode: this split's partial sums, reduced by wgrad_reduce_kernel
            for (int ti = 0; ti < p.TC; ++ti) {
                const int tap = colmode ? 3 * ti + int(blockIdx.y) : tap0 + ti;
                float* dst = p.partial + ((size_t(split) * p.ntaps + tap) * p.Cout + (o0 + row)) * p.Cin + c0;
                for (int cc = 0; cc < p.NC; cc += 16) {
                    const int tcol = colmode ? ((cc >> 6) * 3 + ti) * 64 + (cc & 63) : ti * p.NC + cc;
                    uint32_t v[16];
                    tmem_ld16(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(tcol), v);
                    tmem_ld_wait();
                    if (valid) {
#pragma unroll
                        for (int j = 0; j < 16; j += 4)
                            *reinterpret_cast<float4*>(dst + cc + j) =
                                make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                            __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                    }
                }
            }
        }
        if (k_end > k_begin && do_bias) {  // every column of the ones-accumulator holds sum_pixels dY[pix][o]
            uint32_t v[16];
            tmem_ld16(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(p.TC * p.NC), v);
            tmem_ld_wait();
            if (valid) {
                atomicAdd(p.dbias + o0 + row, __uint_as_float(v[0]));
                if (p.dbias2) atomicAdd(p.dbias2 + o0 + row, __uint_as_float(v[0]));
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, p.tmem_cols);
}

// dweight[o][c][tap] = sum_split partial[split][tap][o][c], deterministic (fixed summation tree).
// grid (ceil(n/32), ntaps), block 256 = 32 consecutive (o,c) elements x 8 split lanes: every warp reads whole
// 128-byte rows of one split, 8 splits are in flight per block.
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ partial,
                                                           float* __restrict__ dweight, int nsplit, int ntaps,
                                                           size_t n) {
    pdl_entry();
    __shared__ float red[8][33];
    const int el = threadIdx.x & 31, lane8 = threadIdx.x >> 5;
    const size_t e = size_t(blockIdx.x) * 32 + el;
    const int tap = blockIdx.y;
    float s0 = 0.f, s1 = 0.f;
    if (e < n) {
        int sp = lane8;
        for (; sp + 8 < nsplit; sp += 16) {
            s0 += partial[(size_t(sp) * ntaps + tap) * n + e];
            s1 += partial[(size_t(sp + 8) * ntaps + tap) * n + e];
        }
        if (sp < nsplit) s0 += partial[(size_t(sp) * ntaps + tap) * n + e];
    }
    red[lane8][el] = s0 + s1;
    __syncthreads();
    if (lane8 == 0 && e < n) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][el];
        dweight[e * ntaps + tap] = t;
    }
}

// dw[o][c][tap] = acc[tap][o][c]; acc = 0.  grid (ceil(max_elems / 256), n_entries), block 288 = 32 (o,c) pairs x 9 taps,
// eight 32-element chunks per block: reads are 9 coalesced 128-byte rows per chunk, the write one contiguous 1152-byte
// run.  (One chunk per block -- 26 880 blocks of 1.1 KB for a bucket -- cost 16 us per launch in ncu, mostly block
// scheduling; skipping the kernel altogether bought 0.04 ms of the step, profiles/r02_skip_experiments.txt.)
__global__ void __launch_bounds__(288) wgrad_finalize_kernel(const WgradFinalizeEntry* __restrict__ table) {
    pdl_entry();
    const WgradFinalizeEntry e = table[blockIdx.y];
    const size_t n = size_t(e.Cout) * e.Cin;
    __shared__ float t[2][9][33];
    const int el = threadIdx.x & 31, tap = threadIdx.x >> 5;  // 9 warps: warp = tap
    const int i = threadIdx.x;                                 // output run: (element i / 9, tap i % 9)
    const int oe = i / 9, ot = i - oe * 9;
#pragma unroll 1
    for (int k = 0; k < 8; ++k) {
        const size_t e0 = (size_t(blockIdx.x) * 8 + k) * 32;
        if (e0 >= n) break;  // (uniform over the block)
        float(*tk)[33] = t[k & 1];
        if (e0 + el < n) {
            float* src = e.acc + size_t(tap) * n + e0 + el;
            tk[tap][el] = *src;
            *src = 0.f;
        }
        __syncthreads();  // (double-buffered tile: one barrier per chunk)
        if (e0 + oe < n) e.dw[e0 * 9 + i] = tk[ot][oe];
    }
}

// =====================================================================================================
// host side
// =====================================================================================================
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !ptr) {
            fprintf(stderr, "[unet_b200] cuTensorMapEncodeTiled unavailable (%d)\n", int(e));
            return nullptr;
        }
        fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

int make_act_map(CUtensorMap* m, const __nv_bfloat16* x, int C, int ld, int W, int H, int B, int TW, int TH, int TB) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return -10;
    if ((reinterpret_cast<uintptr_t>(x) & 15) || (ld % 8) != 0) return -11;
    cuuint64_t dims[4] = {cuuint64_t(C), cuuint64_t(W), cuuint64_t(H), cuuint64_t(B)};
    cuuint64_t strides[3] = {cuuint64_t(ld) * 2, cuuint64_t(W) * ld * 2, cuuint64_t(H) * W * ld * 2};
    cuuint32_t box[4] = {64, cuuint32_t(TW), cuuint32_t(TH), cuuint32_t(TB)};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<__nv_bfloat16*>(x), dims, strides, box, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        fprintf(stderr, "[unet_b200] cuTensorMapEncodeTiled(act C=%d ld=%d W=%d H=%d B=%d box=%d,%d,%d) -> %d\n", C, ld,
                W, H, B, TW, TH, TB, int(r));
        return -12;
    }
    return 0;
}

int make_bf16_map_2d(CUtensorMap* m, const __nv_bfloat16* base, int cols, int rows, int ld, int box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return -10;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld % 8) != 0) return -13;
    cuuint64_t dims[2] = {cuuint64_t(cols), cuuint64_t(rows)};
    cuuint64_t strides[1] = {cuuint64_t(ld) * 2};
    cuuint32_t box[2] = {64, cuuint32_t(box_rows)};
    cuuint32_t es[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(base), dims, strides, box, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        fprintf(stderr, "[unet_b200] cuTensorMapEncodeTiled(2d cols=%d rows=%d ld=%d box_rows=%d) -> %d\n", cols, rows,
                ld, box_rows, int(r));
        return -14;
    }
    return 0;
}

static int next_pow2(int v) {
    int r = 1;
    while (r < v) r <<= 1;
    return r;
}
static int ceil_div_i(int a, int b) { return (a + b - 1) / b; }

static constexpr int kBarrierBytes = 256;

int igemm_epi_plan(IgemmEpiParams* e, const ConvEpilogue& ep, int Cout) {
    *e = IgemmEpiParams{};
    e->bias = ep.bias, e->bias2 = ep.bias2, e->rowvec = ep.rowvec, e->residual = ep.residual;
    e->ldr = ep.ldr ? ep.ldr : Cout;
    e->out = ep.out, e->ldo = ep.ldo ? ep.ldo : Cout, e->out_mode = ep.out_mode;
    e->stats = ep.stats;
    e->gn_x = ep.gn_x, e->gn_ldx = ep.gn_ldx, e->gn_chsum = ep.gn_chsum, e->gn_gamma = ep.gn_gamma;
    e->gn_beta = ep.gn_beta, e->gn_S = ep.gn_S, e->gn_silu = ep.gn_silu;
    if (ep.stats || ep.gn_x) {
        if ((ep.stats && ep.gn_x) || ep.out_mode != OUT_NHWC_BF16) return -15;
        if (ep.gn_x) {
            if (ep.residual || !ep.gn_chsum || !ep.gn_gamma || !ep.gn_beta || !ep.gn_S || ep.gn_groups < 1 ||
                Cout % ep.gn_groups)
                return -15;
            if ((ep.gn_ldx % 8) != 0 || (reinterpret_cast<uintptr_t>(ep.gn_x) & 15)) return -15;
            e->gn_cpg = Cout / ep.gn_groups;
        }
    }
    if (e->out_mode != OUT_NCHW_F32) {
        const int esz = e->out_mode == OUT_NHWC_BF16 ? 2 : 4;
        if ((e->ldo * esz) % 16 != 0 || (reinterpret_cast<uintptr_t>(e->out) & 15)) return -6;
    }
    if (e->residual && ((e->ldr % 8) != 0 || (reinterpret_cast<uintptr_t>(e->residual) & 15))) return -7;
    if (e->bias && (reinterpret_cast<uintptr_t>(e->bias) & 15)) return -8;
    if (e->bias2 && (reinterpret_cast<uintptr_t>(e->bias2) & 15)) return -8;
    if (e->rowvec && ((reinterpret_cast<uintptr_t>(e->rowvec) & 15) || (Cout % 4) != 0)) return -8;
    return 0;
}

int igemm_conv_plan(IgemmConvParams* p, const ConvSegDesc* segs, int nseg, int B, int H, int W, int Cout,
                    const ConvEpilogue& ep) {
    memset(p, 0, sizeof(*p));
    if (nseg < 1 || nseg > 2) return -1;
    if (Cout % 16 != 0) return -2;
    // pixel tile first (needed to count CTAs)
    p->TW = W < 128 ? W : 128;
    p->TH = H < 128 / p->TW ? H : 128 / p->TW;
    if (p->TH < 1) p->TH = 1;
    p->TB = B < 128 / (p->TW * p->TH) ? B : 128 / (p->TW * p->TH);
    if (p->TB < 1) p->TB = 1;
    p->tiles_w = ceil_div_i(W, p->TW);
    p->tiles_h = ceil_div_i(H, p->TH);
    p->tiles_b = ceil_div_i(B, p->TB);
    const int pix_tiles = p->tiles_w * p->tiles_h * p->tiles_b;
    // output-channel tile: the largest divisor of Cout that is a multiple of 16 and <= 256 -- but small problems
    // (8x8 / 16x16 layers) would then run on a handful of SMs, each limited by its own L2->SMEM bandwidth, so BN is
    // lowered (not below 64) until there are ~128 CTAs.
    const bool gn_hook = ep.stats || ep.gn_x;
    int BN = 0;
    for (int cand = 256; cand >= 16; cand -= 16)
        if (Cout % cand == 0 && (!gn_hook || cand % 32 == 0)) {
            if (!BN) BN = cand;
            if (cand < 64) break;
            BN = cand;
            if (pix_tiles * (Cout / cand) >= 128) break;
        }
    if (!BN) return -2;
    p->nseg = nseg;
    p->B = B, p->H = H, p->W = W, p->Cout = Cout, p->BN = BN;
    // Two MMA streams for grids of at most one CTA per SM (see igemm_conv_body); both accumulators within 256 TMEM
    // columns so that a weight-gradient CTA of the side stream still finds room.
    p->nacc = 1;
    {
        int nkb = 0;
        for (int s = 0; s < nseg; ++s) nkb += segs[s].ntaps * ceil_div_i(segs[s].Cin, 64);
        if (pix_tiles * (Cout / BN) <= 148 && BN % 32 == 0 && BN <= 128 && nkb >= 4) p->nacc = 2;
    }
    p->tmem_cols = next_pow2(p->nacc * BN < 32 ? 32 : p->nacc * BN);
    p->a_bytes = uint32_t(64 * p->TW * p->TH * p->TB * 2);
    p->b_bytes = uint32_t(64 * BN * 2);
    p->stage_bytes = 16384u + ((p->b_bytes + 1023u) & ~1023u);
    // Two CTAs per SM when possible (one CTA's epilogue overlaps the other's main loop): <= ~110 KiB each.
    // (the smem tail -- barriers, staged addends, GroupNorm constants and reduction scratch -- comes off the budget)
    const int tb_guess = (128 / (p->TW * p->TH)) < 1 ? 1 : 128 / (p->TW * p->TH);
    const uint32_t tail = 1024u + uint32_t(kBarrierBytes) +
                          uint32_t((ep.rowvec ? tb_guess : 1) + (ep.gn_x ? 4 * tb_guess : 0) + (gn_hook ? 8 : 0)) *
                              uint32_t(BN) * 4u;
    int stages = int((113u * 1024u - tail) / p->stage_bytes);
    if (stages < 3) stages = int((227u * 1024u - tail) / p->stage_bytes);
    if (stages > kMaxStages) stages = kMaxStages;
    if (stages < 2) return -3;
    if (p->nacc == 2) {
        // One CTA per SM: the ring may use more than the two-CTA budget (200 KiB; at 128 KiB a wgrad CTA of the
        // side stream still fits beside it).  Measured round 2 (ms per step): with ONE producer warp 128 / 160 /
        // 200 KiB all gave 5.09-5.10; with the second producer warp 5.02 / 4.99 / 4.975 -- default 200.  Stages of
        // TWO K blocks sharing one barrier pair (both issuers on every stage) were slower -- 890 cycles per pair of K
        // blocks in the phase trace against 2 x 322 -- and were removed again.  What bounds the main loop of these
        // layers is the TMA stream itself: the phase trace with the MMAs switched off (UB_TRACE_MODE=1) takes as long
        // as the full kernel (~77 B/clk/SM for the 4-D halo boxes), the MMA stream alone 35 % less.
        int s2 = int((200u * 1024u - tail) / p->stage_bytes);
        if (s2 > kMaxStages) s2 = kMaxStages;
        if (s2 > stages) stages = s2;
    }
    if (p->nacc == 2 && (stages & 1)) {
        // Two issuers need an EVEN ring: with an odd one the owner of a stage alternates, an issuer skips every other
        // phase of a full barrier, and a parity wait that comes one whole phase early passes immediately (this was a
        // rare hang).  One CTA per SM here, so the ring may grow a stage (kept <= 128 KiB beside a wgrad CTA).
        if (size_t(stages + 1) * p->stage_bytes + tail <= 128u * 1024u && stages + 1 <= kMaxStages)
            stages += 1;
        else
            stages -= 1;
    }
    p->stages = stages;
    for (int s = 0; s < nseg; ++s) {
        const ConvSegDesc& d = segs[s];
        if (d.ntaps != 9 && d.ntaps != 1) return -4;
        if (d.Cin % 8 != 0) return -5;
        int r = make_act_map(&p->seg[s].tmA, d.x, d.Cin, d.ldx, W, H, B, p->TW, p->TH, p->TB);
        if (r) return r;
        r = make_bf16_map_2d(&p->seg[s].tmW, d.wp, d.Cin, d.ntaps * Cout, d.Cin, BN);
        if (r) return r;
        p->seg[s].cblocks = ceil_div_i(d.Cin, 64);
        p->seg[s].ntaps = d.ntaps;
        p->seg[s].wp = d.wp, p->seg[s].Cin = d.Cin;
    }
    // the hooks' tiling conditions: 32-column chunks, and the 32 pixels a warp reduces over lie in one image
    if (gn_hook && (BN % 32 != 0 || ((p->TW * p->TH) % 32 != 0 && p->TB > 1))) return -15;
    int r = igemm_epi_plan(&p->epi, ep, Cout);
    if (r) return r;
    p->ncomb = ep.rowvec ? p->TB : 1;
    p->ngimg = ep.gn_x ? p->TB : 0;
    p->nred = gn_hook ? 8 : 0;
    {
        // tensor-core statistics + TMA output store (IgemmConvParams::ms) for the plain stats hook on full
        // 128-pixel tiles of one or two whole images with a 64- or 128-channel N tile, one or two MMA streams
        // (measured round 2: 5.015 ms per step with, 5.043 with the shuffle-reduce statistics; measured, removed)
        const bool full_tiles = W % p->TW == 0 && H % p->TH == 0 && p->TW * p->TH * p->TB == 128;
        // (TMEM: the accumulators, or one Gram matrix per image of the tile if more, then 64 columns of sums.  Against
        // the staged-Y*Y version this moves two shapes: a two-image tile at BN 128 with one MMA stream (320 > 256
        // columns: 8x8 layers at batches of ~150-255 per GPU) now takes the shuffle statistics, and one at BN 64 with
        // one stream allocates 256 columns instead of 128.  Neither occurs in the default B = 32 step.)
        const size_t need = size_t(BN / 64 + 1) * 16384;  // Y atoms and the ones tile in the dead stages
        const int gcols = (p->TB > p->nacc ? p->TB : p->nacc) * BN + 64;
        if (ep.stats && !ep.gn_x && ep.out_mode == OUT_NHWC_BF16 && (BN == 64 || BN == 128) &&
            p->nacc <= 2 && (p->TB == 1 || (p->TB == 2 && (p->TW * p->TH) == 64)) && full_tiles &&
            need <= size_t(p->stages) * p->stage_bytes && gcols <= (p->nacc == 1 ? 256 : 512) &&
            make_act_map(&p->tmO, reinterpret_cast<const __nv_bfloat16*>(ep.out), Cout, p->epi.ldo, W, H, B, p->TW,
                         p->TH, p->TB) == 0) {
            p->ms = 1;
            p->tmem_cols = next_pow2(gcols);
        }
        // ms == 2, store-only: a conv without any hook whose output is an NHWC bf16 tensor leaves through the same staged
        // tile + TMA store (any whole-tile shape, N tiles of 64 .. 256 channels)
        if (!p->ms && !gn_hook && ep.out_mode == OUT_NHWC_BF16 && BN % 64 == 0 &&
            p->nacc <= 2 && full_tiles && size_t(BN / 64) * 16384 <= size_t(p->stages) * p->stage_bytes &&
            make_act_map(&p->tmO, reinterpret_cast<const __nv_bfloat16*>(ep.out), Cout, p->epi.ldo, W, H, B, p->TW,
                         p->TH, p->TB) == 0)
            p->ms = 2;
    }
    if (size_t(p->ncomb + 4 * p->ngimg + p->nred) * BN * sizeof(float) > 24576) return -9;  // smem tail budget
    if (size_t(p->stages) * p->stage_bytes + 1024 + kBarrierBytes +
            size_t(p->ncomb + 4 * p->ngimg + p->nred) * BN * sizeof(float) > size_t(227) * 1024)
        return -3;
    return 0;
}

void igemm_init() {
    static bool done = false;
    if (done) return;
    cudaFuncSetAttribute(igemm_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(227 * 1024));
    cudaFuncSetAttribute(igemm_conv2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(227 * 1024));
    cudaFuncSetAttribute(igemm_conv_ms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(227 * 1024));
    cudaFuncSetAttribute(igemm_conv2_ms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(227 * 1024));
    cudaFuncSetAttribute(igemm_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(227 * 1024));
    done = true;
}

int igemm_conv_launch(const IgemmConvParams& p, cudaStream_t st) {
    igemm_init();
    const size_t smem = size_t(p.stages) * p.stage_bytes + 1024 + kBarrierBytes +
                        size_t(p.ncomb + 4 * p.ngimg + p.nred) * p.BN * sizeof(float);
    dim3 grid(p.tiles_w * p.tiles_h * p.tiles_b, p.Cout / p.BN);
    auto kern = p.nacc == 2 ? igemm_conv2_kernel : igemm_conv_kernel;
    if (p.ms) kern = p.nacc == 2 ? igemm_conv2_ms_kernel : igemm_conv_ms_kernel;
    launch_pdl(kern, dim3(grid), dim3(kConvThreads), smem, st, p);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)  // a failed launch must never pass silently (the output would simply be stale)
        fprintf(stderr, "[unet_b200] igemm_conv launch failed: %s (grid %u x %u, smem %zu, BN %d, stages %d)\n",
                cudaGetErrorString(e), grid.x, grid.y, smem, p.BN, p.stages);
    return int(e);
}

size_t igemm_wgrad_partial_floats(int Cin, int Cout, int ntaps, int nsplit) {
    return size_t(nsplit) * ntaps * Cout * Cin;
}

static int wgrad_plan_common(IgemmWgradParams* p, const __nv_bfloat16* dy, int ldy, const __nv_bfloat16* x, int ldx,
                             int B, int H, int W, int Cin, int Cout, int ntaps, float* partial,
                             size_t partial_cap_floats, int sm_count, bool acc_mode, bool bias) {
    memset(p, 0, sizeof(*p));
    if (ntaps != 9 && ntaps != 1) return -4;
    if (Cin % 64 != 0 || Cout % 64 != 0) return -5;
    p->B = B, p->H = H, p->W = W, p->Cin = Cin, p->Cout = Cout, p->ntaps = ntaps;
    // boxes may overhang the image (TMA zero-fills), they must hold exactly KP pixels
    // K tile = KP pixels per stage.  128 halves the number of TMA issues and barrier round trips per byte (the single
    // producer thread was the pacing resource at KP = 64); 64 is kept for operands whose tiles would not fit.
    int KP = size_t(B) * H * W < 256 ? 64 : 128;
    p->MO = (Cout % 128 == 0) ? 128 : 64;
    p->TC = ntaps == 9 ? 3 : 1;
    // TMEM: TC * NC columns <= 512
    p->NC = (Cin % 128 == 0) ? 128 : 64;
    const int a_atoms = p->MO / 64, b_atoms = p->NC / 64;
    // Column mode (3x3 layers): a CTA owns a filter COLUMN and takes its three dy taps from
    // one halo box of TH + 2 image rows per 64-channel atom instead of three boxes of TH rows -- the main loop runs at
    // the chip-wide L2 -> shared-memory rate, so bytes are time: the activation operand shrinks to
    // (KP + 2 TW TB) / (3 KP) = 0.67 of its size at 64x64, 0.5 at 32x32, 0.42 at 16x16 and 8x8.
    // (halo windows must start on the 8-pixel swizzle atom: image rows of the tile >= 8 pixels, i.e. W > 4; narrower
    // 3x3 layers and 1x1 layers run row mode.  Row mode for every 3x3 layer: measured, removed,
    // profiles/r02n_wgrad_colmode.txt)
    p->colmode = (ntaps == 9 && next_pow2(W) >= 8) ? 1 : 0;
    for (;;) {
        p->KP = KP;
        p->TW = next_pow2(W) < KP ? next_pow2(W) : KP;
        p->TH = next_pow2(H) < KP / p->TW ? next_pow2(H) : KP / p->TW;
        p->TB = KP / (p->TW * p->TH);
        p->hatom = uint32_t((p->TH + 2) * p->TW * p->TB) * 128u;  // one halo box (a multiple of 1 KiB: TW % 8 == 0)
        p->stage_bytes = p->colmode ? uint32_t(a_atoms) * uint32_t(KP) * 128u + uint32_t(b_atoms) * p->hatom
                                    : uint32_t(a_atoms + p->TC * b_atoms) * uint32_t(KP) * 128u;
        // two stages of the chosen tile must fit beside the epilogue's needs
        if (KP == 128 && size_t(2) * p->stage_bytes > size_t(160) * 1024) {
            KP = 64;
            continue;
        }
        break;
    }
    p->lg_img = 0;
    while ((1 << p->lg_img) < p->TW * p->TH) ++p->lg_img;
    p->tiles_w = ceil_div_i(W, p->TW);
    p->tiles_h = ceil_div_i(H, p->TH);
    p->tiles_b = ceil_div_i(B, p->TB);
    p->tmem_cols = next_pow2(p->TC * p->NC + (bias ? 16 : 0) < 32 ? 32 : p->TC * p->NC + (bias ? 16 : 0));
    if (p->tmem_cols > 512) return -3;
    p->tx_bytes = p->stage_bytes;
    int stages = int((96u * 1024u) / p->stage_bytes);
    if (stages < 2) stages = 2;
    if (stages > kMaxStages) stages = kMaxStages;
    if (size_t(stages) * p->stage_bytes > 220u * 1024u) return -3;
    p->stages = stages;
    const int ktiles = p->tiles_w * p->tiles_h * p->tiles_b;
    const int base_ctas = (Cout / p->MO) * (Cin / p->NC) * (ntaps / p->TC);
    // One CTA per SM (a CTA owns the SM's smem and TMEM), and never more CTAs than SMs: a grid of 150 CTAs on 148
    // SMs runs as two waves and doubles the kernel time (ncu r01: 64->64@64x64 took 57 us as (1,3,50)).
    int nsplit = sm_count / base_ctas;
    if (nsplit > ktiles * KP / 256) nsplit = ktiles * KP / 256;  // at least 256 pixels of K per CTA
    if (nsplit < 1) nsplit = 1;
    if (!acc_mode) {
        while (nsplit > 1 && igemm_wgrad_partial_floats(Cin, Cout, ntaps, nsplit) > partial_cap_floats) --nsplit;
        if (igemm_wgrad_partial_floats(Cin, Cout, ntaps, nsplit) > partial_cap_floats) return -9;
    }
    p->nsplit = nsplit;
    p->partial = partial;
    if (bias) p->ones_off = uint32_t(p->stages) * p->stage_bytes;
    int r = make_act_map(&p->tmDY, dy, Cout, ldy, W, H, B, p->TW, p->TH, p->TB);
    if (r) return r;
    r = make_act_map(&p->tmX, x, Cin, ldx, W, H, B, p->TW, p->colmode ? p->TH + 2 : p->TH, p->TB);
    return r;
}

int igemm_wgrad_plan(IgemmWgradParams* p, const __nv_bfloat16* dy, int ldy, const __nv_bfloat16* x, int ldx, int B,
                     int H, int W, int Cin, int Cout, int ntaps, float* partial, size_t partial_cap_floats,
                     int sm_count) {
    return wgrad_plan_common(p, dy, ldy, x, ldx, B, H, W, Cin, Cout, ntaps, partial, partial_cap_floats, sm_count,
                             false, false);
}

int igemm_wgrad_plan_acc(IgemmWgradParams* p, const __nv_bfloat16* dy, int ldy, const __nv_bfloat16* x, int ldx, int B,
                         int H, int W, int Cin, int Cout, int ntaps, float* acc, float* dbias, float* dbias2,
                         int sm_count) {
    int r = wgrad_plan_common(p, dy, ldy, x, ldx, B, H, W, Cin, Cout, ntaps, nullptr, 0, sm_count, true,
                              dbias != nullptr);
    if (r) return r;
    if (!acc || (reinterpret_cast<uintptr_t>(acc) & 15)) return -16;
    p->acc = acc, p->dbias = dbias, p->dbias2 = dbias2;
    // TMA reduce-add epilogue (see the kernel): fp32 map over acc[ntaps * Cout][Cin], box = 32 columns (128 B, the
    // swizzle span) x the MO/4 accumulator rows of one epilogue warp.
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return -10;
    cuuint64_t dims[2] = {cuuint64_t(Cin), cuuint64_t(ntaps) * cuuint64_t(Cout)};
    cuuint64_t strides[1] = {cuuint64_t(Cin) * 4};
    cuuint32_t box[2] = {32, cuuint32_t(p->MO / 4)};
    cuuint32_t es[2] = {1, 1};
    CUresult cr = fn(&p->tmAcc, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, acc, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) {
        fprintf(stderr, "[unet_b200] cuTensorMapEncodeTiled(wgrad acc Cin=%d rows=%d) -> %d\n", Cin, ntaps * Cout,
                int(cr));
        return -17;
    }
    return 0;
}

int igemm_wgrad_finalize(const WgradFinalizeEntry* table_dev, int n_entries, size_t max_elems, cudaStream_t st) {
    if (n_entries < 1) return 0;
    return int(launch_pdl(wgrad_finalize_kernel, dim3(unsigned((max_elems + 255) / 256), unsigned(n_entries)), dim3(288),
                          0, st, table_dev));
}

int igemm_wgrad_launch(const IgemmWgradParams& p, cudaStream_t st) {
    igemm_init();
    // the optional ones tile (8 KiB) sits where the barriers used to be; the barriers move behind it
    const size_t smem = size_t(p.stages) * p.stage_bytes + (p.ones_off ? size_t(p.KP) * 128 : 0) + 1024 + kBarrierBytes;
    dim3 grid((p.Cout / p.MO) * (p.Cin / p.NC), p.ntaps / p.TC, p.nsplit);
    launch_pdl(igemm_wgrad_kernel, dim3(grid), dim3(kWgradThreads), smem, st, p);
    return int(cudaGetLastError());
}

int igemm_wgrad_reduce(const IgemmWgradParams& p, float* dweight, cudaStream_t st) {
    const size_t n = size_t(p.Cout) * p.Cin;
    launch_pdl(wgrad_reduce_kernel, dim3(dim3(unsigned((n + 31) / 32), p.ntaps)), dim3(256), 0, st, p.partial, dweight, p.nsplit, p.ntaps,
                                                                               n);
    return int(cudaGetLastError());
}

}  // namespace ub
