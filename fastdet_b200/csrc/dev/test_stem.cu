// test_stem.cu — developer harness for conv_stem (not part of the shipped library).
// check: the fused stem against (a) a double-precision CPU loop on sampled outputs (all border pixels + random interior ones)
//        and (b) the two-kernel path (conv0_ws + conv_halo<32, 2>) element by element;
// time : both paths at batch 64, 416x416 (and 608x608).      Usage: test_stem [check|time|all]
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../conv_halo.h"
#include "../conv_block.h"
#include "../conv_stem.h"
#include "../conv_tc.h"
#include "../kernels.h"
#include "../options.h"

using namespace fd;

#define CK(x)                                                                              \
    do {                                                                                   \
        cudaError_t e_ = (x);                                                              \
        if (e_ != cudaSuccess) {                                                           \
            printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
            exit(2);                                                                       \
        }                                                                                  \
    } while (0)

static uint32_t rng_state = 777;
static uint32_t urand() { rng_state = rng_state * 1664525u + 1013904223u; return rng_state >> 8; }
static float frand() { return (urand() & 0xFFFF) / 65536.0f - 0.5f; }
static float bf16r(float x) { return __bfloat162float(__float2bfloat16(x)); }

struct Net {
    int n, h, w, ho, wo, pad_hi;
    std::vector<uint8_t> frames;
    std::vector<float> w1, b1, w2, b2;  // w1 [3][3][3][32] fp32; w2 [64][9*32] (bf16-rounded values)
    float alpha = 0.1f;
    uint8_t* d_frames = nullptr;
    float *d_w1 = nullptr, *d_b1 = nullptr;
    __nv_bfloat16 *d_w2 = nullptr, *d_mid = nullptr, *d_out_ref = nullptr, *d_out = nullptr;
};

static void make_net(Net& N, int n, int h, int w, int pad_hi) {
    N.n = n; N.h = h; N.w = w; N.pad_hi = pad_hi;
    N.ho = (h + 1 + pad_hi - 3) / 2 + 1; N.wo = (w + 1 + pad_hi - 3) / 2 + 1;
    N.frames.resize(1ULL * n * h * w * 3);
    for (auto& v : N.frames) v = static_cast<uint8_t>(urand() & 255);
    N.w1.resize(27 * 32); N.b1.resize(32); N.w2.resize(64 * 288); N.b2.resize(64);
    for (auto& v : N.w1) v = frand() * 1.2f;
    for (auto& v : N.b1) v = frand() * 0.5f;
    for (auto& v : N.w2) v = bf16r(frand() * 0.3f);
    for (auto& v : N.b2) v = frand();
    std::vector<__nv_bfloat16> w2b(N.w2.size());
    for (size_t i = 0; i < w2b.size(); ++i) w2b[i] = __float2bfloat16(N.w2[i]);
    CK(cudaMalloc(&N.d_frames, N.frames.size()));
    CK(cudaMalloc(&N.d_w1, N.w1.size() * 4));
    CK(cudaMalloc(&N.d_b1, 256 * 4));
    CK(cudaMalloc(&N.d_w2, w2b.size() * 2));
    CK(cudaMalloc(&N.d_mid, 1ULL * n * h * w * 32 * 2));
    const size_t out_bytes = 1ULL * n * N.ho * N.wo * 64 * 2;
    CK(cudaMalloc(&N.d_out_ref, out_bytes));
    CK(cudaMalloc(&N.d_out, out_bytes));
    CK(cudaMemset(N.d_out, 0xFF, out_bytes));
    CK(cudaMemset(N.d_out_ref, 0xFF, out_bytes));
    CK(cudaMemset(N.d_b1, 0, 256 * 4));
    CK(cudaMemcpy(N.d_frames, N.frames.data(), N.frames.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(N.d_w1, N.w1.data(), N.w1.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(N.d_b1, N.b1.data(), 32 * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(N.d_w2, w2b.data(), w2b.size() * 2, cudaMemcpyHostToDevice));
}
static void free_net(Net& N) {
    cudaFree(N.d_frames); cudaFree(N.d_w1); cudaFree(N.d_b1); cudaFree(N.d_w2); cudaFree(N.d_mid); cudaFree(N.d_out_ref); cudaFree(N.d_out);
}

static int prepare_two(const Net& N, int sms, HaloLaunch* hl) {
    HaloDesc h;
    memset(&h, 0, sizeof(h));
    h.n = N.n; h.hi = N.h; h.wi = N.w; h.cin = 32; h.in_pitch = 32; h.in = N.d_mid;
    h.cout = 64; h.ksize = 3; h.stride = 2; h.pad_lo = 1; h.pad_hi = N.pad_hi;
    h.w = N.d_w2; h.bias_host = N.b2.data(); h.act = 1; h.alpha = N.alpha;
    h.out = N.d_out_ref; h.out_pitch = 64;
    char err[256] = "";
    if (conv_halo_prepare(h, sms, hl, err, sizeof(err))) { printf("halo prepare failed: %s\n", err); return -1; }
    return 0;
}
static int launch_two(const Net& N, const HaloLaunch& hl) {
    if (launch_conv0_u8(N.d_frames, N.d_w1, N.d_b1, N.d_mid, N.n, N.h, N.w, 32, 1, 32, 1, N.alpha, 0, 0)) return -1;
    return conv_halo_launch(hl, 0);
}
static int prepare_stem(const Net& N, int sms, StemLaunch* sl) {
    StemDesc d;
    memset(&d, 0, sizeof(d));
    d.n = N.n; d.h = N.h; d.w = N.w; d.frames = N.d_frames;
    d.c1 = 32; d.w1 = N.d_w1; d.bias1_host = N.b1.data(); d.act1 = 1; d.alpha1 = N.alpha;
    d.c2 = 64; d.pad_hi2 = N.pad_hi; d.w2 = N.d_w2; d.bias2_host = N.b2.data(); d.act2 = 1; d.alpha2 = N.alpha;
    d.out = N.d_out; d.out_pitch = 64;
    char err[256] = "";
    if (conv_stem_prepare(d, sms, sl, err, sizeof(err))) { printf("stem prepare failed: %s\n", err); return -1; }
    return 0;
}

static double leaky(double x, double a) { return x > 0 ? x : x * a; }

static int check_case(const char* name, int n, int h, int w, int pad_hi, int sms) {
    Net N;
    make_net(N, n, h, w, pad_hi);
    HaloLaunch hl;
    StemLaunch sl;
    if (prepare_two(N, sms, &hl) || prepare_stem(N, sms, &sl)) return 1;
    if (launch_two(N, hl)) { printf("%s: two-kernel launch failed: %s\n", name, cudaGetErrorString(cudaGetLastError())); return 1; }
    CK(cudaDeviceSynchronize());
    if (conv_stem_launch(sl, 0)) { printf("%s: stem launch failed: %s\n", name, cudaGetErrorString(cudaGetLastError())); return 1; }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%s: stem kernel failed: %s\n", name, cudaGetErrorString(e)); exit(3); }
    const size_t elems = 1ULL * n * N.ho * N.wo * 64;
    std::vector<__nv_bfloat16> got(elems), two(elems);
    CK(cudaMemcpy(got.data(), N.d_out, elems * 2, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(two.data(), N.d_out_ref, elems * 2, cudaMemcpyDeviceToHost));
    // (b) against the two-kernel path
    size_t differ = 0, big = 0;
    double maxd = 0;
    for (size_t i = 0; i < elems; ++i) {
        const float a = __bfloat162float(got[i]), b = __bfloat162float(two[i]);
        if (!(a == b)) {
            ++differ;
            const double d = fabs(static_cast<double>(a) - b);
            if (!(d <= 0.02 + 0.02 * fabs(b))) { if (big < 5) printf("   vs two-kernel: elem %zu stem %g two %g\n", i, a, b); ++big; }
            if (d > maxd || d != d) maxd = d;
        }
    }
    // (a) against the CPU loop on samples
    std::vector<float> lutf(256), w1r(N.w1.size());
    for (int i = 0; i < 256; ++i) lutf[i] = bf16r(static_cast<float>(static_cast<double>(i) / 255.0));
    for (size_t i = 0; i < w1r.size(); ++i) w1r[i] = bf16r(N.w1[i]);
    auto c1val = [&](int f, int y, int x, int ci) -> double {
        if (y < 0 || y >= h || x < 0 || x >= w) return 0.0;
        double s = 0;
        for (int r = 0; r < 3; ++r)
            for (int q = 0; q < 3; ++q) {
                const int yy = y - 1 + r, xx = x - 1 + q;
                if (yy < 0 || yy >= h || xx < 0 || xx >= w) continue;
                const uint8_t* px = &N.frames[((1ULL * f * h + yy) * w + xx) * 3];
                for (int ch = 0; ch < 3; ++ch) s += static_cast<double>(lutf[px[ch]]) * w1r[((r * 3 + q) * 3 + ch) * 32 + ci];
            }
        return bf16r(static_cast<float>(leaky(s + N.b1[ci], N.alpha)));
    };
    int bad = 0, samples = 0;
    double worst = 0;
    auto check_px = [&](int f, int oy, int ox) {
        double c1[9][32];
        for (int r = 0; r < 3; ++r)
            for (int q = 0; q < 3; ++q)
                for (int ci = 0; ci < 32; ++ci) c1[r * 3 + q][ci] = c1val(f, 2 * oy - 1 + r, 2 * ox - 1 + q, ci);
        for (int co = 0; co < 64; ++co) {
            double s = 0;
            for (int t = 0; t < 9; ++t)
                for (int ci = 0; ci < 32; ++ci) s += c1[t][ci] * N.w2[co * 288 + t * 32 + ci];
            const double ref = leaky(s + N.b2[co], N.alpha);
            const double g = __bfloat162float(got[((1ULL * f * N.ho + oy) * N.wo + ox) * 64 + co]);
            const double err = fabs(g - ref);
            ++samples;
            if (err > worst || err != err) worst = err;
            if (!(err <= 0.02 + 0.01 * fabs(ref))) {
                if (bad < 8) printf("   vs CPU: f %d oy %d ox %d co %d got %g want %g\n", f, oy, ox, co, g, ref);
                ++bad;
            }
        }
    };
    for (int f = 0; f < n; f += (n > 2 ? n - 1 : 1)) {
        for (int ox = 0; ox < N.wo; ++ox) { check_px(f, 0, ox); check_px(f, N.ho - 1, ox); }
        for (int oy = 0; oy < N.ho; ++oy) { check_px(f, oy, 0); check_px(f, oy, N.wo - 1); }
    }
    for (int i = 0; i < 600; ++i) check_px(urand() % n, urand() % N.ho, urand() % N.wo);
    // tile seams: rows / columns around multiples of the 16 x 8 tile
    for (int i = 0; i < 200; ++i) {
        const int oy = std::min(N.ho - 1, static_cast<int>(urand() % ((N.ho + 15) / 16)) * 16 + static_cast<int>(urand() % 2) * 15);
        const int ox = std::min(N.wo - 1, static_cast<int>(urand() % ((N.wo + 7) / 8)) * 8 + static_cast<int>(urand() % 2) * 7);
        check_px(urand() % n, oy, ox);
    }
    const int fail = bad || big;
    printf("%-28s n %d %dx%d pad_hi %d: vs CPU %d samples, %d bad, worst %.4f | vs two-kernel: %zu of %zu differ (max %.4f), %zu beyond tolerance  %s\n",
           name, n, h, w, pad_hi, samples, bad, worst, differ, elems, maxd, big, fail ? "FAIL" : "ok");
    free_net(N);
    return fail ? 1 : 0;
}

static void time_case(int n, int hw, int sms, int debug = 0) {
    Net N;
    make_net(N, n, hw, hw, 1);
    HaloLaunch hl;
    StemLaunch sl;
    if (prepare_two(N, sms, &hl) || prepare_stem(N, sms, &sl)) return;
    sl.p.debug = debug;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    const int reps = 20;
    float ms_two = 0, ms_stem = 0;
    for (int pass = 0; pass < 2; ++pass) {
        for (int i = 0; i < 3; ++i) launch_two(N, hl);
        CK(cudaEventRecord(e0));
        for (int i = 0; i < reps; ++i) launch_two(N, hl);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        CK(cudaEventElapsedTime(&ms_two, e0, e1));
        for (int i = 0; i < 3; ++i) conv_stem_launch(sl, 0);
        CK(cudaEventRecord(e0));
        for (int i = 0; i < reps; ++i) conv_stem_launch(sl, 0);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        CK(cudaEventElapsedTime(&ms_stem, e0, e1));
    }
    CK(cudaDeviceSynchronize());
    {   // one profiled launch: per role, cycles per tile in its loop and in its barrier waits (averaged over the CTAs)
        long long* dprof;
        CK(cudaMalloc(&dprof, sl.grid * 16 * sizeof(long long)));
        CK(cudaMemset(dprof, 0, sl.grid * 16 * sizeof(long long)));
        StemLaunch pl = sl;
        pl.p.prof = dprof;
        conv_stem_launch(pl, 0);
        CK(cudaDeviceSynchronize());
        std::vector<long long> hp(sl.grid * 16);
        CK(cudaMemcpy(hp.data(), dprof, hp.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        double avg[16] = {0};
        for (int b = 0; b < sl.grid; ++b)
            for (int i = 0; i < 16; ++i) avg[i] += static_cast<double>(hp[b * 16 + i]) / sl.grid;
        const double tiles = 1.0 * sl.p.total / sl.grid;
        printf("   cycles/tile  builder: loop %.0f wait in_empty %.0f publish %.0f signal %.0f | mma: loop %.0f wait in_full %.0f acc1_empty %.0f acc2_empty+c1_full %.0f | "
               "epi1(g0): loop %.0f wait c1_empty %.0f acc1_full %.0f | epi2: loop %.0f wait acc2_full %.0f store_read %.0f\n",
               avg[0] / tiles, avg[1] / tiles, avg[2] / tiles, avg[3] / tiles, avg[4] / tiles, avg[5] / tiles, avg[6] / tiles, avg[7] / tiles, avg[8] / tiles, avg[9] / tiles,
               avg[10] / tiles, avg[12] / tiles, avg[13] / tiles, avg[14] / tiles);
        cudaFree(dprof);
    }
    printf("dbg %3d time n %d %dx%d: two kernels %.1f us, stem %.1f us (%.2fx), stem %.1f TFLOP/s algorithmic, out %.0f MB\n", debug, n, hw, hw,
           ms_two * 1000 / reps, ms_stem * 1000 / reps, ms_two / ms_stem, sl.flops / (ms_stem / reps * 1e-3) / 1e12,
           1.0 * n * N.ho * N.wo * 128 / 1e6);
    free_net(N);
}


// ------------------------------------------------------------------------------------------------ conv_block
struct Blk {
    int n, h, w;
    std::vector<float> x, wa, ba, wb, bb;  // bf16-rounded values (biases fp32)
    float alpha = 0.1f;
    __nv_bfloat16 *d_x = nullptr, *d_wa = nullptr, *d_wb = nullptr, *d_mid = nullptr, *d_out_ref = nullptr, *d_out = nullptr;
    float *d_ba = nullptr;
};
static void make_blk(Blk& B, int n, int h, int w) {
    B.n = n; B.h = h; B.w = w;
    B.x.resize(1ULL * n * h * w * 64); B.wa.resize(32 * 64); B.ba.resize(32); B.wb.resize(64 * 288); B.bb.resize(64);
    for (auto& v : B.x) v = bf16r(frand() * 2.f);
    for (auto& v : B.wa) v = bf16r(frand() * 0.4f);
    for (auto& v : B.ba) v = frand() * 0.5f;
    for (auto& v : B.wb) v = bf16r(frand() * 0.3f);
    for (auto& v : B.bb) v = frand();
    auto up = [](const std::vector<float>& v, __nv_bfloat16** d) {
        std::vector<__nv_bfloat16> b(v.size());
        for (size_t i = 0; i < v.size(); ++i) b[i] = __float2bfloat16(v[i]);
        CK(cudaMalloc(d, b.size() * 2));
        CK(cudaMemcpy(*d, b.data(), b.size() * 2, cudaMemcpyHostToDevice));
    };
    up(B.x, &B.d_x); up(B.wa, &B.d_wa); up(B.wb, &B.d_wb);
    CK(cudaMalloc(&B.d_mid, 1ULL * n * h * w * 32 * 2));
    CK(cudaMalloc(&B.d_out_ref, B.x.size() * 2));
    CK(cudaMalloc(&B.d_out, B.x.size() * 2));
    CK(cudaMemset(B.d_out, 0xFF, B.x.size() * 2));
    CK(cudaMalloc(&B.d_ba, 1024 * 4));
    CK(cudaMemset(B.d_ba, 0, 1024 * 4));
    CK(cudaMemcpy(B.d_ba, B.ba.data(), 32 * 4, cudaMemcpyHostToDevice));
}
static void free_blk(Blk& B) { cudaFree(B.d_x); cudaFree(B.d_wa); cudaFree(B.d_wb); cudaFree(B.d_mid); cudaFree(B.d_out_ref); cudaFree(B.d_out); cudaFree(B.d_ba); }

static int prepare_blk_two(const Blk& B, int sms, ConvLaunch* cl, HaloLaunch* hl) {
    ConvDesc d;
    memset(&d, 0, sizeof(d));
    d.n = B.n; d.hi = B.h; d.wi = B.w; d.cin = 64; d.in_pitch = 64; d.in = B.d_x;
    d.cout = 32; d.ksize = 1; d.stride = 1; d.w = B.d_wa; d.bias = B.d_ba; d.bias_host = B.ba.data(); d.act = 1; d.alpha = B.alpha;
    d.out = B.d_mid; d.out_pitch = 32;
    char err[256] = "";
    if (conv_tc_prepare(d, sms, 0, cl, err, sizeof(err))) { printf("1x1 prepare failed: %s\n", err); return -1; }
    HaloDesc h;
    memset(&h, 0, sizeof(h));
    h.n = B.n; h.hi = B.h; h.wi = B.w; h.cin = 32; h.in_pitch = 32; h.in = B.d_mid;
    h.cout = 64; h.ksize = 3; h.stride = 1; h.pad_lo = 1; h.pad_hi = 1;
    h.w = B.d_wb; h.bias_host = B.bb.data(); h.act = 1; h.alpha = B.alpha;
    h.residual = B.d_x; h.res_pitch = 64;
    h.out = B.d_out_ref; h.out_pitch = 64;
    if (conv_halo_prepare(h, sms, hl, err, sizeof(err))) { printf("halo prepare failed: %s\n", err); return -1; }
    return 0;
}
static int prepare_blk(const Blk& B, int sms, BlockLaunch* bl) {
    BlockDesc d;
    memset(&d, 0, sizeof(d));
    d.n = B.n; d.h = B.h; d.w = B.w; d.in = B.d_x; d.in_pitch = 64; d.cin = 64; d.cmid = 32; d.cout = 64;
    d.wa = B.d_wa; d.bias_a_host = B.ba.data(); d.act_a = 1; d.alpha_a = B.alpha;
    d.wb = B.d_wb; d.bias_b_host = B.bb.data(); d.act_b = 1; d.alpha_b = B.alpha;
    d.out = B.d_out; d.out_pitch = 64;
    char err[256] = "";
    if (conv_block_prepare(d, sms, bl, err, sizeof(err))) { printf("block prepare failed: %s\n", err); return -1; }
    return 0;
}

static int check_block(const char* name, int n, int h, int w, int sms) {
    Blk B;
    make_blk(B, n, h, w);
    ConvLaunch cl;
    HaloLaunch hl;
    BlockLaunch bl;
    if (prepare_blk_two(B, sms, &cl, &hl) || prepare_blk(B, sms, &bl)) return 1;
    if (conv_tc_launch(cl, 0) || conv_halo_launch(hl, 0)) { printf("%s: two-kernel launch failed\n", name); return 1; }
    CK(cudaDeviceSynchronize());
    if (conv_block_launch(bl, 0)) { printf("%s: block launch failed: %s\n", name, cudaGetErrorString(cudaGetLastError())); return 1; }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%s: block kernel failed: %s\n", name, cudaGetErrorString(e)); exit(3); }
    const size_t elems = B.x.size();
    std::vector<__nv_bfloat16> got(elems), two(elems);
    CK(cudaMemcpy(got.data(), B.d_out, elems * 2, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(two.data(), B.d_out_ref, elems * 2, cudaMemcpyDeviceToHost));
    size_t differ = 0, big = 0;
    double maxd = 0;
    for (size_t i = 0; i < elems; ++i) {
        const float a = __bfloat162float(got[i]), b = __bfloat162float(two[i]);
        if (!(a == b)) {
            ++differ;
            const double d = fabs(static_cast<double>(a) - b);
            if (!(d <= 0.03 + 0.02 * fabs(b))) { if (big < 5) printf("   vs two-kernel: elem %zu block %g two %g\n", i, a, b); ++big; }
            if (d > maxd || d != d) maxd = d;
        }
    }
    auto midval = [&](int f, int y, int x, int c) -> double {
        if (y < 0 || y >= h || x < 0 || x >= w) return 0.0;
        double s = 0;
        const float* px = &B.x[((1ULL * f * h + y) * w + x) * 64];
        for (int ci = 0; ci < 64; ++ci) s += static_cast<double>(px[ci]) * B.wa[c * 64 + ci];
        return bf16r(static_cast<float>(leaky(s + B.ba[c], B.alpha)));
    };
    int bad = 0, samples = 0;
    double worst = 0;
    auto check_px = [&](int f, int oy, int ox) {
        double mid[9][32];
        for (int r = 0; r < 3; ++r)
            for (int q = 0; q < 3; ++q)
                for (int c = 0; c < 32; ++c) mid[r * 3 + q][c] = midval(f, oy - 1 + r, ox - 1 + q, c);
        for (int co = 0; co < 64; ++co) {
            double s = 0;
            for (int t = 0; t < 9; ++t)
                for (int c = 0; c < 32; ++c) s += mid[t][c] * B.wb[co * 288 + t * 32 + c];
            const size_t o = ((1ULL * f * h + oy) * w + ox) * 64 + co;
            const double ref = leaky(s + B.bb[co], B.alpha) + B.x[o];
            const double g = __bfloat162float(got[o]);
            const double err = fabs(g - ref);
            ++samples;
            if (err > worst || err != err) worst = err;
            if (!(err <= 0.03 + 0.01 * fabs(ref))) {
                if (bad < 8) printf("   vs CPU: f %d oy %d ox %d co %d got %g want %g\n", f, oy, ox, co, g, ref);
                ++bad;
            }
        }
    };
    for (int f = 0; f < n; f += (n > 2 ? n - 1 : 1)) {
        for (int ox = 0; ox < w; ++ox) { check_px(f, 0, ox); check_px(f, h - 1, ox); }
        for (int oy = 0; oy < h; ++oy) { check_px(f, oy, 0); check_px(f, oy, w - 1); }
    }
    for (int i = 0; i < 600; ++i) check_px(urand() % n, urand() % h, urand() % w);
    for (int i = 0; i < 200; ++i) {
        const int oy = std::min(h - 1, static_cast<int>(urand() % ((h + 15) / 16)) * 16 + static_cast<int>(urand() % 2) * 15);
        const int ox = std::min(w - 1, static_cast<int>(urand() % ((w + 7) / 8)) * 8 + static_cast<int>(urand() % 2) * 7);
        check_px(urand() % n, oy, ox);
    }
    const int fail = bad || big;
    printf("block %-22s n %d %dx%d: vs CPU %d samples, %d bad, worst %.4f | vs two-kernel: %zu of %zu differ (max %.4f), %zu beyond tolerance  %s\n",
           name, n, h, w, samples, bad, worst, differ, elems, maxd, big, fail ? "FAIL" : "ok");
    free_blk(B);
    return fail ? 1 : 0;
}

static void time_block(int n, int hw, int sms, int debug = 0) {
    Blk B;
    make_blk(B, n, hw, hw);
    ConvLaunch cl;
    HaloLaunch hl;
    BlockLaunch bl;
    if (prepare_blk_two(B, sms, &cl, &hl) || prepare_blk(B, sms, &bl)) return;
    bl.p.debug = debug;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    const int reps = 20;
    float ms_two = 0, ms_blk = 0;
    for (int pass = 0; pass < 2; ++pass) {
        for (int i = 0; i < 3; ++i) { conv_tc_launch(cl, 0); conv_halo_launch(hl, 0); }
        CK(cudaEventRecord(e0));
        for (int i = 0; i < reps; ++i) { conv_tc_launch(cl, 0); conv_halo_launch(hl, 0); }
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        CK(cudaEventElapsedTime(&ms_two, e0, e1));
        for (int i = 0; i < 3; ++i) conv_block_launch(bl, 0);
        CK(cudaEventRecord(e0));
        for (int i = 0; i < reps; ++i) conv_block_launch(bl, 0);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        CK(cudaEventElapsedTime(&ms_blk, e0, e1));
    }
    CK(cudaDeviceSynchronize());
    {
        long long* dprof;
        CK(cudaMalloc(&dprof, bl.grid * 16 * sizeof(long long)));
        CK(cudaMemset(dprof, 0, bl.grid * 16 * sizeof(long long)));
        BlockLaunch pl = bl;
        pl.p.prof = dprof;
        conv_block_launch(pl, 0);
        CK(cudaDeviceSynchronize());
        std::vector<long long> hp(bl.grid * 16);
        CK(cudaMemcpy(hp.data(), dprof, hp.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        double avg[16] = {0};
        for (int b = 0; b < bl.grid; ++b)
            for (int i = 0; i < 16; ++i) avg[i] += static_cast<double>(hp[b * 16 + i]) / bl.grid;
        const double tiles = 1.0 * bl.p.total / bl.grid;
        printf("   cycles/tile  builder: loop %.0f wait in_empty %.0f | mma: loop %.0f wait in_full %.0f acca_empty %.0f accb_empty+mid_full %.0f | "
               "epiA(b0): loop %.0f wait mid_empty %.0f acca_full %.0f | epiB: loop %.0f wait accb_full %.0f store_read %.0f\n",
               avg[0] / tiles, avg[1] / tiles, avg[4] / tiles, avg[5] / tiles, avg[6] / tiles, avg[7] / tiles, avg[8] / tiles, avg[9] / tiles,
               avg[10] / tiles, avg[12] / tiles, avg[13] / tiles, avg[14] / tiles);
        cudaFree(dprof);
    }
    printf("dbg %3d block n %d %dx%d: two kernels %.1f us, block %.1f us (%.2fx)\n", debug, n, hw, hw, ms_two * 1000 / reps, ms_blk * 1000 / reps, ms_two / ms_blk);
    free_blk(B);
}

int main(int argc, char** argv) {
    const char* mode = argc > 1 ? argv[1] : "all";
    int dev = 0, sms = 148;
    CK(cudaSetDevice(dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    char err[256] = "";
    if (conv_tc_init(err, sizeof(err))) { printf("conv_tc_init: %s\n", err); return 2; }
    if (kernels_init() || conv_halo_init() || conv_stem_init() || conv_block_init()) { printf("kernel init failed: %s\n", cudaGetErrorString(cudaGetLastError())); return 2; }
    int fails = 0;
    if (!strcmp(mode, "check") || !strcmp(mode, "all")) {
        fails += check_case("one tile row", 1, 128, 128, 1, sms);
        fails += check_case("416", 2, 416, 416, 1, sms);
        fails += check_case("ragged 150x140", 3, 150, 140, 1, sms);
        fails += check_case("odd rows 131x132", 2, 131, 132, 1, sms);
        fails += check_case("pad (1,0) 160x192", 2, 160, 192, 0, sms);
        fails += check_case("many tiles per CTA", 12, 224, 224, 1, sms);
        fails += check_block("one tile row", 1, 64, 64, sms);
        fails += check_block("208", 2, 208, 208, sms);
        fails += check_block("ragged 75x70", 3, 75, 70, sms);
        fails += check_block("many tiles per CTA", 12, 112, 112, sms);
        printf("check: %d failing case(s)\n", fails);
    }
    if (!strcmp(mode, "time") || !strcmp(mode, "all")) {
        time_case(64, 416, sms);
        time_case(16, 416, sms);
        time_case(32, 608, sms);
        time_block(64, 208, sms);
        time_block(32, 304, sms);
    }
    if (!strcmp(mode, "blk")) {
        int f2 = check_block("one tile row", 1, 64, 64, sms) + check_block("208", 2, 208, 208, sms) + check_block("ragged 75x70", 3, 75, 70, sms) +
                 check_block("many tiles per CTA", 12, 112, 112, sms);
        printf("check: %d failing case(s)\n", f2);
        for (int dbg : {0, 1, 2, 12, 16}) time_block(64, 208, sms, dbg);
        return f2 ? 1 : 0;
    }
    if (!strcmp(mode, "probe"))
        for (int dbg : {0, 12, 1, 2, 16}) time_case(64, 416, sms, dbg);
    return fails ? 1 : 0;
}
