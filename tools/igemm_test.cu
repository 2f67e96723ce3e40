// Standalone GPU harness for the tcgen05 implicit-GEMM kernels (development tool, not part of the library).
//   ./igemm_test [quick | plans]
// Checks igemm_conv (fprop, 1x1, two-segment, all epilogue modes) and igemm_wgrad against a CPU reference
// computed from the same bf16-rounded operands, probes UMMA descriptor start-address/base_offset behaviour,
// checks that both conv planners accept and reject the same epilogues (`plans`: only that table),
// and prints CUDA-event timings.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

#include "../unet.cu_b200/csrc/igemm.cuh"
#include "../unet.cu_b200/csrc/ptx.cuh"

using namespace ub;

#define CK(x)                                                                          \
    do {                                                                               \
        cudaError_t e_ = (x);                                                          \
        if (e_ != cudaSuccess) {                                                       \
            printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
            exit(2);                                                                   \
        }                                                                              \
    } while (0)

static float bf16r(float f) { return __bfloat162float(__float2bfloat16(f)); }

struct Rng {
    std::mt19937 g;
    std::normal_distribution<float> nd{0.f, 1.f};
    explicit Rng(int s) : g(s) {}
    float n() { return nd(g); }
};

static int g_fail = 0;

// ------------------------------------------------------------------------------------------ conv test
// x NHWC [B,H,W,Cin], w reference layout [Cout][Cin][ntaps]
static void cpu_conv_point(const std::vector<float>& x, const std::vector<float>& w, int B, int H, int W, int Cin,
                           int Cout, int ntaps, int b, int h, int ww, int o, double* acc) {
    double s = 0;
    for (int tap = 0; tap < ntaps; ++tap) {
        int dy = ntaps == 9 ? tap / 3 - 1 : 0, dx = ntaps == 9 ? tap % 3 - 1 : 0;
        int hh = h + dy, wx = ww + dx;
        if (hh < 0 || hh >= H || wx < 0 || wx >= W) continue;
        const float* xp = &x[((size_t(b) * H + hh) * W + wx) * Cin];
        const float* wp = &w[size_t(o) * Cin * ntaps + tap];
        for (int c = 0; c < Cin; ++c) s += double(xp[c]) * double(wp[size_t(c) * ntaps]);
    }
    *acc += s;
}

static bool test_conv(int B, int H, int W, int Cin, int Cout, int ntaps, int Cin2, int out_mode, bool use_bias,
                      bool use_rowvec, bool use_res, int nsample, int reps, bool halo = false) {
    Rng rng(1234 + Cin + Cout + H);
    size_t npix = size_t(B) * H * W;
    std::vector<float> x(npix * Cin), w(size_t(Cout) * Cin * ntaps), x2, w2, bias(Cout), rowvec(size_t(B) * Cout),
        res(npix * Cout);
    float ws = 1.f / sqrtf(float(ntaps * Cin));
    for (auto& v : x) v = bf16r(rng.n());
    for (auto& v : w) v = bf16r(rng.n() * ws);
    for (auto& v : bias) v = rng.n();
    for (auto& v : rowvec) v = rng.n();
    for (auto& v : res) v = bf16r(rng.n());
    if (Cin2) {
        x2.resize(npix * Cin2);
        w2.resize(size_t(Cout) * Cin2);
        for (auto& v : x2) v = bf16r(rng.n());
        for (auto& v : w2) v = bf16r(rng.n() / sqrtf(float(Cin2)));
    }
    // pack
    std::vector<__nv_bfloat16> xb(x.size()), wpk(size_t(ntaps) * Cout * Cin), x2b(x2.size()), w2pk(w2.size()),
        resb(res.size());
    for (size_t i = 0; i < x.size(); ++i) xb[i] = __float2bfloat16(x[i]);
    for (size_t i = 0; i < res.size(); ++i) resb[i] = __float2bfloat16(res[i]);
    for (int t = 0; t < ntaps; ++t)
        for (int o = 0; o < Cout; ++o)
            for (int c = 0; c < Cin; ++c)
                wpk[(size_t(t) * Cout + o) * Cin + c] = __float2bfloat16(w[(size_t(o) * Cin + c) * ntaps + t]);
    for (size_t i = 0; i < x2.size(); ++i) x2b[i] = __float2bfloat16(x2[i]);
    for (size_t i = 0; i < w2.size(); ++i) w2pk[i] = __float2bfloat16(w2[i]);

    __nv_bfloat16 *dx, *dw, *dx2 = nullptr, *dw2 = nullptr, *dres;
    float *dbias, *drow;
    void* dout;
    size_t out_elems = npix * Cout;
    size_t out_bytes = out_elems * (out_mode == OUT_NHWC_BF16 ? 2 : 4);
    CK(cudaMalloc(&dx, xb.size() * 2));
    CK(cudaMalloc(&dw, wpk.size() * 2));
    CK(cudaMalloc(&dres, resb.size() * 2));
    CK(cudaMalloc(&dbias, Cout * 4));
    CK(cudaMalloc(&drow, rowvec.size() * 4));
    CK(cudaMalloc(&dout, out_bytes));
    CK(cudaMemcpy(dx, xb.data(), xb.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dw, wpk.data(), wpk.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dres, resb.data(), resb.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dbias, bias.data(), Cout * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(drow, rowvec.data(), rowvec.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemset(dout, 0xFF, out_bytes));
    if (Cin2) {
        CK(cudaMalloc(&dx2, x2b.size() * 2));
        CK(cudaMalloc(&dw2, w2pk.size() * 2));
        CK(cudaMemcpy(dx2, x2b.data(), x2b.size() * 2, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dw2, w2pk.data(), w2pk.size() * 2, cudaMemcpyHostToDevice));
    }
    ConvSegDesc segs[2] = {{dx, Cin, Cin, dw, ntaps}, {dx2, Cin2, Cin2, dw2, 1}};
    ConvEpilogue ep;
    ep.bias = use_bias ? dbias : nullptr;
    ep.rowvec = use_rowvec ? drow : nullptr;
    ep.residual = use_res ? dres : nullptr;
    ep.out = dout;
    ep.out_mode = out_mode;
    float* dstats = nullptr;
    if (getenv("UB_TEST_STATS") && out_mode == OUT_NHWC_BF16 && Cout % 32 == 0) {  // time the GroupNorm-statistics hook
        CK(cudaMalloc(&dstats, size_t(B) * Cout * 2 * sizeof(float)));
        CK(cudaMemset(dstats, 0, size_t(B) * Cout * 2 * sizeof(float)));
        ep.stats = dstats;
    }
    IgemmConvParams p;
    IgemmRowsParams ph;
    int r = halo ? igemm_rows_plan(&ph, segs, Cin2 ? 2 : 1, B, H, W, Cout, ep, 148)
                 : igemm_conv_plan(&p, segs, Cin2 ? 2 : 1, B, H, W, Cout, ep);
    if (r) {
        printf("conv plan failed %d\n", r);
        g_fail++;
        return false;
    }
    auto launch = [&]() { return halo ? igemm_rows_launch(ph, 0) : igemm_conv_launch(p, 0); };
#ifdef UB_TRACE
    igemm_trace_set_mode(0);
#endif
    r = launch();
    cudaError_t e = cudaDeviceSynchronize();
    if (r || e != cudaSuccess) {
        printf("conv launch failed r=%d e=%s\n", r, cudaGetErrorString(e));
        exit(3);
    }
    std::vector<uint8_t> hout(out_bytes);
    CK(cudaMemcpy(hout.data(), dout, out_bytes, cudaMemcpyDeviceToHost));

    // verify on a sample of output points (all points if small)
    std::mt19937 g(7);
    size_t total = out_elems;
    bool all = total <= size_t(nsample);
    size_t ncheck = all ? total : nsample;
    double max_err = 0, max_ref = 0;
    int bad = 0;
    for (size_t i = 0; i < ncheck; ++i) {
        size_t idx = all ? i : (size_t(g()) * 2654435761ull + g()) % total;
        int o = idx % Cout;
        size_t pix = idx / Cout;
        int ww = pix % W, h = (pix / W) % H, b = pix / (size_t(W) * H);
        double acc = 0;
        cpu_conv_point(x, w, B, H, W, Cin, Cout, ntaps, b, h, ww, o, &acc);
        if (Cin2) cpu_conv_point(x2, w2, B, H, W, Cin2, Cout, 1, b, h, ww, o, &acc);
        if (use_bias) acc += bias[o];
        if (use_rowvec) acc += rowvec[size_t(b) * Cout + o];
        if (use_res) acc += res[pix * Cout + o];
        float got;
        if (out_mode == OUT_NHWC_BF16)
            got = __bfloat162float(reinterpret_cast<__nv_bfloat16*>(hout.data())[pix * Cout + o]);
        else if (out_mode == OUT_NHWC_F32)
            got = reinterpret_cast<float*>(hout.data())[pix * Cout + o];
        else
            got = reinterpret_cast<float*>(hout.data())[((size_t(b) * Cout + o) * H + h) * W + ww];
        double err = fabs(double(got) - acc);
        double tol = (out_mode == OUT_NHWC_BF16 ? 1e-2 : 2e-3) * (1.0 + fabs(acc));
        if (!(err <= tol)) {
            if (bad < 5) printf("   mismatch b=%d h=%d w=%d o=%d got=%f ref=%f\n", b, h, ww, o, got, acc);
            bad++;
        }
        if (err > max_err) max_err = err;
        if (fabs(acc) > max_ref) max_ref = fabs(acc);
    }
    // timing
    float ms = 0;
    if (reps > 0) {
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
#ifdef UB_TRACE
        if (getenv("UB_TRACE_MODE")) igemm_trace_set_mode(atoi(getenv("UB_TRACE_MODE")));  // (results are garbage)
#endif
        for (int i = 0; i < 3; ++i) launch();
        cudaEventRecord(e0);
        for (int i = 0; i < reps; ++i) launch();
        cudaEventRecord(e1);
        CK(cudaEventSynchronize(e1));
        cudaEventElapsedTime(&ms, e0, e1);
        ms /= reps;
    }
#ifdef UB_TRACE
    if (!halo && reps > 0) igemm_trace_dump(p.tiles_w * p.tiles_h * p.tiles_b * (p.Cout / p.BN), 1.965);
    if (halo && reps > 0) igemm_rows_trace_dump(std::min(ph.num_tiles, 148), ph.num_tiles);
#endif
    if (dstats) cudaFree(dstats);
    double flops = 2.0 * npix * Cout * (double(ntaps) * Cin + Cin2);
    printf("%s B%d %dx%d %d->%d taps%d seg2=%d mode%d b%d r%d s%d | BN=%d stages=%d | checked %zu bad %d max_err %.3g "
           "(max_ref %.3g) | %.4f ms %.1f TFLOP/s  %s\n",
           halo ? "ROWS" : "conv", B, H, W, Cin, Cout, ntaps, Cin2, out_mode, use_bias, use_rowvec, use_res,
           halo ? ph.BN : p.BN, halo ? ph.w_stages : p.stages, ncheck, bad,
           max_err, max_ref, ms, ms > 0 ? flops / ms * 1e-9 : 0.0, bad ? "FAIL" : "ok");
    if (bad) g_fail++;
    cudaFree(dx), cudaFree(dw), cudaFree(dres), cudaFree(dbias), cudaFree(drow), cudaFree(dout);
    if (dx2) cudaFree(dx2), cudaFree(dw2);
    return bad == 0;
}

// ------------------------------------------------------------------------------------------ planner contract
// Both conv planners must accept and reject the same epilogues, with the same codes, at a shape both kernels take
// (B 2, 64->64 @ 64x64, 3x3).  Nothing is launched: the buffers only have to exist and be aligned.
static void test_plan_contract() {
    const int B = 2, H = 64, W = 64, C = 64;
    const size_t act = size_t(B) * H * W * C, vec = size_t(B) * C * 2;
    __nv_bfloat16 *x, *wp, *res, *gx, *out;
    float *bias, *stats, *chsum, *gamma, *beta, *S;
    CK(cudaMalloc(&x, act * 2));
    CK(cudaMalloc(&wp, size_t(9) * C * C * 2));
    CK(cudaMalloc(&res, act * 2));
    CK(cudaMalloc(&gx, act * 2));
    CK(cudaMalloc(&out, act * 4));  // room for an fp32 output
    CK(cudaMalloc(&bias, 64 * 4));  // (bias, second bias, row vector: the planners only read the addresses)
    CK(cudaMalloc(&stats, vec * 4));
    CK(cudaMalloc(&chsum, vec * 4));
    CK(cudaMalloc(&gamma, C * 4));
    CK(cudaMalloc(&beta, C * 4));
    CK(cudaMalloc(&S, vec * 4));
    const ConvSegDesc seg = {x, C, C, wp, 9};
    ConvEpilogue plain;
    plain.bias = bias, plain.bias2 = bias, plain.rowvec = bias, plain.residual = res, plain.out = out;
    ConvEpilogue st;
    st.bias = bias, st.residual = res, st.out = out, st.stats = stats;
    ConvEpilogue gn;
    gn.out = out, gn.gn_x = gx, gn.gn_ldx = C, gn.gn_chsum = chsum, gn.gn_gamma = gamma, gn.gn_beta = beta;
    gn.gn_S = S, gn.gn_silu = 1;
    struct Case {
        const char* name;
        ConvEpilogue ep;
        int want;
    };
    std::vector<Case> cases = {{"bias + bias2 + rowvec + residual", plain, 0}, {"statistics hook", st, 0},
                               {"gn-bwd hook", gn, 0}};
    auto add = [&](const char* name, ConvEpilogue ep, int want) { cases.push_back({name, ep, want}); };
    {
        ConvEpilogue e = gn;
        e.stats = stats;
        add("stats with gn_x", e, -15);
        e = gn, e.residual = res;
        add("gn_x with residual", e, -15);
        e = gn, e.gn_chsum = nullptr;
        add("gn_x without statistics", e, -15);
        e = gn, e.gn_gamma = nullptr;
        add("gn_x without gamma", e, -15);
        e = gn, e.gn_beta = nullptr;
        add("gn_x without beta", e, -15);
        e = gn, e.gn_S = nullptr;
        add("gn_x without S", e, -15);
        e = gn, e.gn_groups = 24;
        add("gn_groups not dividing Cout", e, -15);
        e = gn, e.gn_ldx = 68;
        add("gn_ldx % 8 != 0", e, -15);
        e = gn, e.gn_x = gx + 1;
        add("misaligned gn_x", e, -15);
        e = st, e.out_mode = OUT_NHWC_F32;
        add("stats with fp32 output", e, -15);
        e = gn, e.out_mode = OUT_NCHW_F32;
        add("gn_x with fp32 output", e, -15);
        e = plain, e.bias = bias + 1;
        add("misaligned bias", e, -8);
        e = plain, e.bias2 = bias + 1;
        add("misaligned bias2", e, -8);
        e = plain, e.rowvec = bias + 1;
        add("misaligned rowvec", e, -8);
        e = plain, e.residual = res + 1;
        add("misaligned residual", e, -7);
        e = plain, e.ldr = 68;
        add("ldr % 8 != 0", e, -7);
        e = plain, e.out = out + 1;
        add("misaligned output", e, -6);
        e = plain, e.out = out + 1, e.out_mode = OUT_NHWC_F32;
        add("misaligned fp32 output", e, -6);
        e = plain, e.ldo = 68;
        add("ldo % 8 != 0", e, -6);
    }
    printf("== planner contract (B%d %dx%d %d->%d taps9) ==\n", B, H, W, C, C);
    for (const Case& c : cases) {
        IgemmConvParams p;
        IgemmRowsParams pr;
        const int rc = igemm_conv_plan(&p, &seg, 1, B, H, W, C, c.ep);
        const int rr = igemm_rows_plan(&pr, &seg, 1, B, H, W, C, c.ep, 148);
        const bool ok = rc == c.want && rr == c.want;
        printf("  %-34s conv %4d  rows %4d  (want %3d)  %s\n", c.name, rc, rr, c.want, ok ? "ok" : "FAIL");
        if (!ok) g_fail++;
    }
    cudaFree(x), cudaFree(wp), cudaFree(res), cudaFree(gx), cudaFree(out), cudaFree(bias);
    cudaFree(stats), cudaFree(chsum), cudaFree(gamma), cudaFree(beta), cudaFree(S);
}

// ------------------------------------------------------------------------------------------ wgrad test
static bool test_wgrad(int B, int H, int W, int Cin, int Cout, int ntaps, int nsample, int reps) {
    Rng rng(99 + Cin + Cout + H);
    size_t npix = size_t(B) * H * W;
    std::vector<float> x(npix * Cin), dy(npix * Cout);
    for (auto& v : x) v = bf16r(rng.n());
    for (auto& v : dy) v = bf16r(rng.n());
    std::vector<__nv_bfloat16> xb(x.size()), dyb(dy.size());
    for (size_t i = 0; i < x.size(); ++i) xb[i] = __float2bfloat16(x[i]);
    for (size_t i = 0; i < dy.size(); ++i) dyb[i] = __float2bfloat16(dy[i]);
    __nv_bfloat16 *dx_, *ddy;
    float *dpart, *ddw;
    size_t cap = size_t(64) << 20;  // 64M floats = 256 MB
    CK(cudaMalloc(&dx_, xb.size() * 2));
    CK(cudaMalloc(&ddy, dyb.size() * 2));
    CK(cudaMalloc(&dpart, cap * 4));
    CK(cudaMalloc(&ddw, size_t(Cout) * Cin * ntaps * 4));
    CK(cudaMemcpy(dx_, xb.data(), xb.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ddy, dyb.data(), dyb.size() * 2, cudaMemcpyHostToDevice));
    IgemmWgradParams p;
    int r = igemm_wgrad_plan(&p, ddy, Cout, dx_, Cin, B, H, W, Cin, Cout, ntaps, dpart, cap, 148);
    if (r) {
        printf("wgrad plan failed %d\n", r);
        g_fail++;
        return false;
    }
    r = igemm_wgrad_launch(p, 0);
    r |= igemm_wgrad_reduce(p, ddw, 0);
    cudaError_t e = cudaDeviceSynchronize();
    if (r || e != cudaSuccess) {
        printf("wgrad launch failed r=%d e=%s\n", r, cudaGetErrorString(e));
        exit(3);
    }
    std::vector<float> hdw(size_t(Cout) * Cin * ntaps);
    CK(cudaMemcpy(hdw.data(), ddw, hdw.size() * 4, cudaMemcpyDeviceToHost));
    std::mt19937 g(11);
    size_t total = hdw.size();
    bool all = total <= size_t(nsample);
    size_t ncheck = all ? total : nsample;
    int bad = 0;
    double max_err = 0, max_ref = 0;
    for (size_t i = 0; i < ncheck; ++i) {
        size_t idx = all ? i : (size_t(g()) * 2654435761ull + g()) % total;
        int tap = idx % ntaps;
        int c = (idx / ntaps) % Cin;
        int o = idx / (size_t(ntaps) * Cin);
        int dyy = ntaps == 9 ? tap / 3 - 1 : 0, dxx = ntaps == 9 ? tap % 3 - 1 : 0;
        double acc = 0;
        for (int b = 0; b < B; ++b)
            for (int h = 0; h < H; ++h) {
                int hh = h + dyy;
                if (hh < 0 || hh >= H) continue;
                for (int w = 0; w < W; ++w) {
                    int wx = w + dxx;
                    if (wx < 0 || wx >= W) continue;
                    acc += double(dy[((size_t(b) * H + h) * W + w) * Cout + o]) *
                           double(x[((size_t(b) * H + hh) * W + wx) * Cin + c]);
                }
            }
        double err = fabs(double(hdw[idx]) - acc);
        double tol = 2e-3 * (1.0 + fabs(acc)) + 1e-3 * sqrt(double(npix));
        if (!(err <= tol)) {
            if (bad < 5) printf("   mismatch o=%d c=%d tap=%d got=%f ref=%f\n", o, c, tap, hdw[idx], acc);
            bad++;
        }
        if (err > max_err) max_err = err;
        if (fabs(acc) > max_ref) max_ref = fabs(acc);
    }
    float ms = 0, ms_red = 0;
    if (reps > 0) {
        cudaEvent_t e0, e1, e2;
        cudaEventCreate(&e0), cudaEventCreate(&e1), cudaEventCreate(&e2);
        for (int i = 0; i < 3; ++i) igemm_wgrad_launch(p, 0);
        cudaEventRecord(e0);
        for (int i = 0; i < reps; ++i) igemm_wgrad_launch(p, 0);
        cudaEventRecord(e1);
        for (int i = 0; i < reps; ++i) igemm_wgrad_reduce(p, ddw, 0);
        cudaEventRecord(e2);
        CK(cudaEventSynchronize(e2));
        cudaEventElapsedTime(&ms, e0, e1);
        cudaEventElapsedTime(&ms_red, e1, e2);
        ms /= reps, ms_red /= reps;
    }
    double flops = 2.0 * npix * Cout * double(ntaps) * Cin;
    printf("wgrad B%d %dx%d %d->%d taps%d | %s MO=%d NC=%d TC=%d split=%d stages=%d | checked %zu bad %d max_err %.3g "
           "(max_ref %.3g) | %.4f ms (+%.4f reduce) %.1f TFLOP/s  %s\n",
           B, H, W, Cin, Cout, ntaps, p.colmode ? "col" : "row", p.MO, p.NC, p.TC, p.nsplit, p.stages, ncheck, bad, max_err,
           max_ref, ms, ms_red,
           ms > 0 ? flops / ms * 1e-9 : 0.0, bad ? "FAIL" : "ok");
    if (bad) g_fail++;
    // accumulate mode (the trainer's): every CTA adds its tile into acc[tap][o][c] with TMA reduce-add boxes --
    // compared with the two-pass result above, element by element
    float *dacc, *dbias;
    CK(cudaMalloc(&dacc, hdw.size() * 4));
    CK(cudaMalloc(&dbias, size_t(Cout) * 4));
    CK(cudaMemset(dacc, 0, hdw.size() * 4));
    CK(cudaMemset(dbias, 0, size_t(Cout) * 4));
    IgemmWgradParams pa;
    r = igemm_wgrad_plan_acc(&pa, ddy, Cout, dx_, Cin, B, H, W, Cin, Cout, ntaps, dacc, dbias, nullptr, 148);
    if (r) {
        printf("wgrad acc plan failed %d\n", r);
        g_fail++;
        return false;
    }
    r = igemm_wgrad_launch(pa, 0);
    e = cudaDeviceSynchronize();
    if (r || e != cudaSuccess) {
        printf("wgrad acc launch failed r=%d e=%s\n", r, cudaGetErrorString(e));
        exit(3);
    }
    std::vector<float> hacc(hdw.size()), hb(Cout);
    CK(cudaMemcpy(hacc.data(), dacc, hacc.size() * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(hb.data(), dbias, hb.size() * 4, cudaMemcpyDeviceToHost));
    int bad2 = 0;
    double me = 0;
    for (int tap = 0; tap < ntaps; ++tap)
        for (int o = 0; o < Cout; ++o)
            for (int c = 0; c < Cin; ++c) {
                const double a = hacc[(size_t(tap) * Cout + o) * Cin + c], b = hdw[(size_t(o) * Cin + c) * ntaps + tap];
                const double err = fabs(a - b);
                if (err > me) me = err;
                if (!(err <= 1e-4 * (1.0 + fabs(b)) + 2e-5 * sqrt(double(npix)))) {
                    if (bad2 < 5) printf("   acc mismatch tap=%d o=%d c=%d got=%f two-pass=%f\n", tap, o, c, a, b);
                    bad2++;
                }
            }
    int badb = 0;
    for (int o = 0; o < Cout; ++o) {  // bias gradient = column sums of dY
        double sref = 0;
        for (size_t px = 0; px < npix; ++px) sref += dy[px * Cout + o];
        if (!(fabs(hb[o] - sref) <= 1e-3 * (1.0 + fabs(sref)) + 1e-4 * sqrt(double(npix)))) {
            if (badb < 3) printf("   bias mismatch o=%d got=%f ref=%f\n", o, hb[o], sref);
            badb++;
        }
    }
    float msa = 0;
    if (reps > 0) {
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0), cudaEventCreate(&e1);
        for (int i = 0; i < 3; ++i) igemm_wgrad_launch(pa, 0);
        cudaEventRecord(e0);
        for (int i = 0; i < reps; ++i) igemm_wgrad_launch(pa, 0);
        cudaEventRecord(e1);
        CK(cudaEventSynchronize(e1));
        cudaEventElapsedTime(&msa, e0, e1);
        msa /= reps;
    }
    printf("   acc mode (TMA reduce-add) max |acc - two-pass| %.3g bad %d bias bad %d | %.4f ms %.1f TFLOP/s  %s\n", me,
           bad2, badb, msa, msa > 0 ? flops / msa * 1e-9 : 0.0, (bad2 || badb) ? "FAIL" : "ok");
    if (bad2 || badb) g_fail++;
    cudaFree(dacc), cudaFree(dbias);
    cudaFree(dx_), cudaFree(ddy), cudaFree(dpart), cudaFree(ddw);
    return bad == 0;
}

// ------------------------------------------------------------------------------------------ descriptor probe
// One CTA. A_big: 256 rows x 64 bf16 (128-byte rows, SWIZZLE_128B written by TMA). Bm: 64 rows x 64 bf16 (K-major).
// mode 0: A K-major,  D[m][n] = sum_k A_big[m + j][k] * Bm[n][k]        (start address + j*128 B)
// mode 1: A MN-major, D[m][n] = sum_{k<64} A_big[k + j][m] * Bm[n][k]   (M = 64, start address + j*128 B)
struct ProbeParams {
    CUtensorMap tmA, tmB;
    int mode, j, base_offset;
    float* out;  // [128][64]
};
__global__ void __launch_bounds__(128) probe_kernel(const __grid_constant__ ProbeParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;             // 256 * 128 = 32 KB
    uint8_t* sB = smem + 32768;     // 64 * 128 = 8 KB
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 32768 + 8192);
    uint64_t* bar2 = bar + 1;
    uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_init(bar2, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        tmem_alloc(slot, 64);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tm = *slot;
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, 32768 + 8192);
        tma_load_2d(sA, &p.tmA, bar, 0, 0);
        tma_load_2d(sB, &p.tmB, bar, 0, 0);
        mbar_wait(bar, 0);
        tc_fence_after();
        const uint32_t a0 = smem_u32(sA) + p.j * 128;
        const uint32_t b0 = smem_u32(sB);
        if (p.mode == 0) {
            const uint32_t idesc = make_idesc_bf16(128, 64, 0, 0);
            for (int k = 0; k < 4; ++k) {
                uint64_t dA = make_smem_desc_sw128(a0 + k * 32, 16, 1024, p.base_offset);
                uint64_t dB = make_smem_desc_sw128(b0 + k * 32, 16, 1024);
                umma_bf16(tm, dA, dB, idesc, k != 0);
            }
        } else {
            const uint32_t idesc = make_idesc_bf16(64, 64, 1, 0);
            for (int k = 0; k < 4; ++k) {
                uint64_t dA = make_smem_desc_sw128(a0 + k * 2048, 8192, 1024, p.base_offset);
                uint64_t dB = make_smem_desc_sw128(b0 + k * 32, 16, 1024);
                umma_bf16(tm, dA, dB, idesc, k != 0);
            }
        }
        umma_commit(bar2);
    }
    mbar_wait(bar2, 0);
    tc_fence_after();
    for (int c0 = 0; c0 < 64; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(tm + (uint32_t(warp * 32) << 16) + c0, v);
        tmem_ld_wait();
        for (int i = 0; i < 16; ++i) p.out[(warp * 32 + lane) * 64 + c0 + i] = __uint_as_float(v[i]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 64);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static void run_probe() {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres));
    EncodeTiledFn fn = (EncodeTiledFn)ptr;
    Rng rng(5);
    std::vector<float> A(256 * 64), Bm(64 * 64);
    for (auto& v : A) v = bf16r(rng.n());
    for (auto& v : Bm) v = bf16r(rng.n());
    std::vector<__nv_bfloat16> Ab(A.size()), Bb(Bm.size());
    for (size_t i = 0; i < A.size(); ++i) Ab[i] = __float2bfloat16(A[i]);
    for (size_t i = 0; i < Bm.size(); ++i) Bb[i] = __float2bfloat16(Bm[i]);
    __nv_bfloat16 *dA, *dB;
    float* dout;
    CK(cudaMalloc(&dA, Ab.size() * 2));
    CK(cudaMalloc(&dB, Bb.size() * 2));
    CK(cudaMalloc(&dout, 128 * 64 * 4));
    CK(cudaMemcpy(dA, Ab.data(), Ab.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dB, Bb.data(), Bb.size() * 2, cudaMemcpyHostToDevice));
    ProbeParams p;
    {
        cuuint64_t dims[2] = {64, 256};
        cuuint64_t strides[1] = {128};
        cuuint32_t box[2] = {64, 256};
        cuuint32_t es[2] = {1, 1};
        CUresult r = fn(&p.tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dA, dims, strides, box, es,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        cuuint64_t dimsb[2] = {64, 64};
        cuuint32_t boxb[2] = {64, 64};
        CUresult r2 = fn(&p.tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dB, dimsb, strides, boxb, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r || r2) {
            printf("probe: tensor map encode failed %d %d\n", int(r), int(r2));
            return;
        }
    }
    p.out = dout;
    CK(cudaFuncSetAttribute(probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    std::vector<float> hout(128 * 64);
    for (int mode = 0; mode < 2; ++mode) {
        for (int j : {0, 1, 2, 3, 5, 8, 9, 66}) {
            for (int bo_kind = 0; bo_kind < 2; ++bo_kind) {
                p.mode = mode, p.j = j, p.base_offset = bo_kind ? (j & 7) : 0;
                if (bo_kind == 1 && (j & 7) == 0) continue;
                probe_kernel<<<1, 128, 48 * 1024, 0>>>(p);
                cudaError_t e = cudaDeviceSynchronize();
                if (e != cudaSuccess) {
                    printf("probe mode=%d j=%d bo=%d: CUDA error %s\n", mode, j, p.base_offset, cudaGetErrorString(e));
                    exit(4);
                }
                CK(cudaMemcpy(hout.data(), dout, hout.size() * 4, cudaMemcpyDeviceToHost));
                int M = mode == 0 ? 128 : 64;
                int bad = 0;
                double maxerr = 0;
                for (int m = 0; m < M; ++m)
                    for (int n = 0; n < 64; ++n) {
                        double acc = 0;
                        for (int k = 0; k < 64; ++k)
                            acc += mode == 0 ? double(A[(m + j) * 64 + k]) * Bm[n * 64 + k]
                                             : double(A[(k + j) * 64 + m]) * Bm[n * 64 + k];
                        int lane_row = mode == 0 ? m : (m % 16) + 32 * (m / 16);
                        double err = fabs(hout[lane_row * 64 + n] - acc);
                        if (err > 1e-2 * (1 + fabs(acc))) bad++;
                        if (err > maxerr) maxerr = err;
                    }
                printf("probe mode=%s j=%2d base_offset=%d : %s (bad %d, max_err %.3g)\n",
                       mode == 0 ? "A-Kmajor " : "A-MNmajor", j, p.base_offset, bad ? "MISMATCH" : "match", bad,
                       maxerr);
            }
        }
    }
    cudaFree(dA), cudaFree(dB), cudaFree(dout);
}

int main(int argc, char** argv) {
    bool quick = argc > 1 && !strcmp(argv[1], "quick");
    if (argc > 8 && !strcmp(argv[1], "shape")) {  // shape B H W Cin Cout halo reps  (single case, for ncu)
        int B = atoi(argv[2]), H = atoi(argv[3]), W = atoi(argv[4]), Cin = atoi(argv[5]), Cout = atoi(argv[6]);
        test_conv(B, H, W, Cin, Cout, 9, 0, OUT_NHWC_BF16, true, true, false, 2000, atoi(argv[8]), atoi(argv[7]) != 0);
        return g_fail ? 1 : 0;
    }
    if (argc > 9 && !strcmp(argv[1], "conv")) {  // conv B H W Cin Cout ntaps rows reps  (single timed case, no hooks / addends)
        test_conv(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6]), atoi(argv[7]), 0,
                  OUT_NHWC_BF16, false, false, false, 2000, atoi(argv[9]), atoi(argv[8]) != 0);
        return g_fail ? 1 : 0;
    }
    if (argc > 1 && !strcmp(argv[1], "plans")) {
        test_plan_contract();
        return g_fail ? 1 : 0;
    }
    if (argc > 7 && !strcmp(argv[1], "wgrad")) {  // wgrad B H W Cin Cout reps
        test_wgrad(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6]), 9, 200, atoi(argv[7]));
        return g_fail ? 1 : 0;
    }
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("device: %s, %d SMs, cc %d.%d\n", prop.name, prop.multiProcessorCount, prop.major, prop.minor);

    const bool wgrad_only = argc > 1 && !strcmp(argv[1], "wgradonly");  // only the weight-gradient cases (timed)
    if (wgrad_only) goto wgrad_tests;
    printf("== descriptor probe ==\n");
    run_probe();
    test_plan_contract();

    printf("== conv (fprop / 1x1 / fused) ==\n");
    // tiny shapes first: every output checked
    test_conv(2, 8, 8, 64, 64, 9, 0, OUT_NHWC_F32, false, false, false, 1 << 20, 0);
    test_conv(2, 16, 16, 64, 64, 9, 0, OUT_NHWC_F32, true, false, false, 1 << 20, 0);
    test_conv(2, 16, 16, 128, 64, 9, 0, OUT_NHWC_BF16, true, true, true, 1 << 20, 0);
    test_conv(3, 8, 8, 64, 128, 1, 0, OUT_NCHW_F32, true, false, false, 1 << 20, 0);
    test_conv(2, 16, 16, 64, 192, 9, 128, OUT_NHWC_BF16, true, true, false, 1 << 20, 0);
    test_conv(1, 12, 20, 72, 48, 9, 0, OUT_NHWC_F32, true, false, false, 1 << 20, 0);  // ragged everything
    test_conv(2, 32, 32, 64, 576, 1, 0, OUT_NHWC_BF16, true, false, false, 200000, 0);  // qkv-like (3 N tiles)
    if (!quick) {
        int reps = 20;
        test_conv(32, 64, 64, 64, 64, 9, 0, OUT_NHWC_BF16, true, true, false, 20000, reps);
        test_conv(32, 64, 64, 192, 64, 9, 0, OUT_NHWC_BF16, true, false, false, 20000, reps);
        test_conv(32, 64, 64, 192, 64, 9, 0, OUT_NCHW_F32, true, false, false, 20000, reps);
        test_conv(32, 32, 32, 128, 128, 9, 0, OUT_NHWC_BF16, true, true, false, 20000, reps);
        test_conv(32, 32, 32, 320, 128, 9, 320, OUT_NHWC_BF16, true, true, false, 20000, reps);
        test_conv(32, 16, 16, 192, 192, 9, 0, OUT_NHWC_BF16, true, true, false, 20000, reps);
        test_conv(32, 8, 8, 256, 256, 9, 0, OUT_NHWC_BF16, true, true, false, 20000, reps);
        test_conv(32, 8, 8, 512, 256, 9, 512, OUT_NHWC_BF16, true, true, false, 20000, reps);
        test_conv(32, 16, 16, 192, 576, 1, 0, OUT_NHWC_BF16, true, false, false, 20000, reps);
        test_conv(32, 64, 64, 256, 256, 9, 0, OUT_NHWC_BF16, true, false, false, 20000, reps);
        test_conv(32, 64, 64, 512, 512, 9, 0, OUT_NHWC_BF16, true, false, false, 5000, 5);
    }
    printf("== persistent row-tile conv (igemm_rows) ==\n");
    test_conv(1, 32, 32, 64, 64, 9, 0, OUT_NHWC_F32, false, false, false, 1 << 20, 0, true);
    test_conv(2, 32, 32, 64, 64, 9, 0, OUT_NHWC_F32, true, false, false, 1 << 20, 0, true);
    test_conv(2, 64, 64, 128, 64, 9, 0, OUT_NHWC_BF16, true, true, true, 1 << 20, 0, true);
    test_conv(3, 32, 32, 64, 128, 1, 0, OUT_NCHW_F32, true, false, false, 1 << 20, 0, true);
    test_conv(2, 32, 32, 64, 192, 9, 128, OUT_NHWC_BF16, true, true, false, 1 << 20, 0, true);
    test_conv(1, 24, 16, 72, 48, 9, 0, OUT_NHWC_F32, true, false, false, 1 << 20, 0, true);  // ragged H, Cin
    test_conv(5, 16, 16, 192, 192, 9, 0, OUT_NHWC_BF16, true, true, false, 1 << 20, 0, true);
    test_conv(1, 128, 128, 64, 64, 9, 0, OUT_NHWC_BF16, true, false, false, 200000, 0, true);
    if (!quick) {
        int reps = 20;
        test_conv(32, 64, 64, 64, 64, 9, 0, OUT_NHWC_BF16, true, true, false, 20000, reps, true);
        test_conv(32, 64, 64, 128, 64, 9, 0, OUT_NHWC_BF16, true, true, false, 20000, reps, true);
        test_conv(32, 64, 64, 192, 64, 9, 0, OUT_NHWC_BF16, true, false, false, 20000, reps, true);
        test_conv(32, 64, 64, 64, 64, 9, 64, OUT_NHWC_BF16, true, true, false, 20000, reps, true);
        test_conv(32, 64, 64, 64, 128, 9, 0, OUT_NHWC_BF16, true, true, false, 20000, reps, true);
        test_conv(32, 32, 32, 128, 128, 9, 0, OUT_NHWC_BF16, true, true, false, 20000, reps, true);
        test_conv(32, 32, 32, 320, 128, 9, 320, OUT_NHWC_BF16, true, true, false, 20000, reps, true);
        test_conv(32, 32, 32, 64, 128, 9, 64, OUT_NHWC_BF16, true, true, false, 20000, reps, true);
        test_conv(32, 16, 16, 192, 192, 9, 0, OUT_NHWC_BF16, true, true, false, 20000, reps, true);
        test_conv(32, 16, 16, 192, 576, 1, 0, OUT_NHWC_BF16, true, false, false, 20000, reps, true);
        test_conv(32, 64, 64, 256, 256, 9, 0, OUT_NHWC_BF16, true, false, false, 20000, reps, true);
        test_conv(32, 64, 64, 512, 512, 9, 0, OUT_NHWC_BF16, true, false, false, 5000, 5, true);
    }
wgrad_tests:
    // column mode (3x3 layers with W > 4: one halo box per filter column) and row mode (1x1 layers and 3x3 layers with
    // W <= 4: three boxes per filter row); the plan picks the mode from the shape
    printf("== wgrad ==\n");
    test_wgrad(2, 8, 8, 64, 64, 9, 1 << 20, 0);
    test_wgrad(5, 8, 8, 64, 64, 9, 1 << 20, 0);     // two images per K tile, the last tile half outside the batch
    test_wgrad(6, 8, 8, 128, 128, 9, 1 << 20, 0);
    test_wgrad(2, 16, 16, 128, 128, 9, 20000, 0);
    test_wgrad(3, 8, 8, 64, 128, 1, 1 << 20, 0);
    test_wgrad(2, 4, 4, 64, 64, 9, 1 << 20, 0);     // 3x3 row mode
    test_wgrad(3, 4, 2, 128, 64, 9, 1 << 20, 0);
    test_wgrad(4, 3, 3, 64, 128, 9, 1 << 20, 0);
    test_wgrad(2, 12, 20, 64, 64, 9, 1 << 20, 0);
    test_wgrad(3, 20, 12, 64, 64, 9, 1 << 20, 0);
    test_wgrad(4, 16, 16, 192, 64, 9, 20000, 0);
    test_wgrad(2, 32, 32, 64, 128, 9, 20000, 0);
    if (!quick) {
        int reps = 20;
        test_wgrad(32, 64, 64, 64, 64, 9, 400, reps);
        test_wgrad(32, 64, 64, 192, 64, 9, 400, reps);
        test_wgrad(32, 64, 64, 64, 128, 9, 400, reps);
        test_wgrad(32, 32, 32, 128, 128, 9, 400, reps);
        test_wgrad(32, 16, 16, 192, 192, 9, 1000, reps);
        test_wgrad(32, 8, 8, 256, 256, 9, 2000, reps);
        test_wgrad(32, 8, 8, 512, 256, 9, 2000, reps);
        test_wgrad(32, 32, 32, 320, 128, 1, 2000, reps);
        test_wgrad(32, 64, 64, 256, 256, 9, 200, reps);
    }
    printf("== %s (%d failing groups) ==\n", g_fail ? "FAILED" : "ALL OK", g_fail);
    return g_fail ? 1 : 0;
}
