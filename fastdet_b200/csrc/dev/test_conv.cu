// test_conv.cu — developer harness for conv_tc (not part of the shipped library).
// Checks the tcgen05 implicit-GEMM conv (every form: single CTA, CTA pair, swapped, split-K, strips) and the halo-patch
// kernel against a double-precision CPU loop on small shapes and on the production split-K shapes, then times the hot YOLOv3
// layer shapes at batch 64.   Usage: test_conv [check|time|all]
//
// The check holds every output element to the rounding model of tests/compare.py (layer_bound): inputs and weights are
// bf16, so every product is exact in fp32 and the kernel's fp32 sum of K products + bias (+ activation, + residual) is within
// A = 2^-23 * (K + 4) * S of the exact value, S = sum |x w| + |b| (+ |res|); a bf16 output adds half a bf16 step at
// max(|got|, |ref|); the halo kernel's residual form rounds the branch first (+ half a step of the branch); a fused
// MaxPool(2, 2) takes the largest bound in its window.  Split-K cases are marked "splitK" in the case line.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../conv_halo.h"
#include "../conv_tc.h"
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

static uint32_t rng_state = 12345;
static float frand() {
    rng_state = rng_state * 1664525u + 1013904223u;
    return ((rng_state >> 8) & 0xFFFF) / 65536.0f - 0.5f;
}
static float bf16r(float x) { return __bfloat162float(__float2bfloat16(x)); }
// spacing of bf16 numbers at |v| (8 significant bits; subnormal spacing below 2^-126)
static double bf16_ulp(double v) {
    int e;
    frexp(fmax(fabs(v), ldexp(1.0, -126)), &e);
    return ldexp(1.0, e - 8);
}
static const double kU = ldexp(1.0, -23);  // one fp32 addition, relative to the running magnitude (allows truncation)

struct Case {
    const char* name;
    int n, h, w, cin, cout, k, stride, pad_lo, pad_hi, act, residual, fp32, upsample, in_pitch_extra, block_n;
    int pool;  // 1: MaxPool(2, 2) fused into the epilogue (halo-patch kernel only); omitted = 0
};

static int run_case(const Case& c, int num_sms) {
    const int in_pitch = c.cin + c.in_pitch_extra;
    const int ho = (c.h + c.pad_lo + c.pad_hi - c.k) / c.stride + 1;
    const int wo = (c.w + c.pad_lo + c.pad_hi - c.k) / c.stride + 1;
    const long long M = 1LL * c.n * ho * wo;
    const int K = c.k * c.k * c.cin;
    const int out_pitch = c.fp32 ? ((c.cout + 15) / 16) * 16 : c.cout + 8;  // exercise pitch != cout
    const int oh = c.upsample ? 2 * ho : (c.pool ? ho / 2 : ho), ow = c.upsample ? 2 * wo : (c.pool ? wo / 2 : wo);

    std::vector<float> x(1LL * c.n * c.h * c.w * in_pitch), wt(1LL * c.cout * K), bias(1024, 0.f),
        res(c.residual ? M * c.cout : 0);
    for (auto& v : x) v = bf16r(frand() * 2.f);
    for (auto& v : wt) v = bf16r(frand() * 0.25f);
    for (int i = 0; i < c.cout; ++i) bias[i] = frand();
    for (auto& v : res) v = bf16r(frand());

    std::vector<__nv_bfloat16> xb(x.size()), wb(wt.size()), rb(res.size());
    for (size_t i = 0; i < x.size(); ++i) xb[i] = __float2bfloat16(x[i]);
    for (size_t i = 0; i < wt.size(); ++i) wb[i] = __float2bfloat16(wt[i]);
    for (size_t i = 0; i < res.size(); ++i) rb[i] = __float2bfloat16(res[i]);

    __nv_bfloat16 *dx, *dw, *dr = nullptr;
    float* dbias;
    void* dout;
    const size_t out_elems = 1ULL * c.n * oh * ow * out_pitch;
    const size_t out_bytes = out_elems * (c.fp32 ? 4 : 2);
    CK(cudaMalloc(&dx, xb.size() * 2));
    CK(cudaMalloc(&dw, wb.size() * 2));
    CK(cudaMalloc(&dbias, bias.size() * 4));
    CK(cudaMalloc(&dout, out_bytes));
    CK(cudaMemset(dout, 0xFF, out_bytes));
    if (c.residual) {
        CK(cudaMalloc(&dr, rb.size() * 2));
        CK(cudaMemcpy(dr, rb.data(), rb.size() * 2, cudaMemcpyHostToDevice));
    }
    CK(cudaMemcpy(dx, xb.data(), xb.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dw, wb.data(), wb.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dbias, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice));

    ConvDesc d;
    memset(&d, 0, sizeof(d));
    d.n = c.n; d.hi = c.h; d.wi = c.w; d.cin = c.cin; d.in_pitch = in_pitch; d.in = dx;
    d.cout = c.cout; d.ksize = c.k; d.stride = c.stride; d.pad_lo = c.pad_lo; d.pad_hi = c.pad_hi;
    d.w = dw; d.bias = dbias; d.bias_host = bias.data(); d.act = c.act; d.alpha = 0.1f;
    d.residual = dr; d.res_pitch = c.cout;
    d.out = dout; d.out_pitch = out_pitch; d.out_fp32 = c.fp32; d.upsample2x = c.upsample;
    ConvLaunch L;
    memset(&L, 0, sizeof(L));
    char err[256] = {0};
    if (c.block_n == 2048) {  // the halo-patch kernel (conv_halo.cu) on the same problem
        HaloDesc hd;
        memset(&hd, 0, sizeof(hd));
        hd.n = d.n; hd.hi = d.hi; hd.wi = d.wi; hd.cin = d.cin; hd.in_pitch = d.in_pitch; hd.in = d.in;
        hd.cout = d.cout; hd.ksize = d.ksize; hd.stride = d.stride; hd.pad_lo = d.pad_lo; hd.pad_hi = d.pad_hi;
        hd.w = d.w; hd.bias_host = d.bias_host; hd.act = d.act; hd.alpha = d.alpha;
        hd.residual = d.residual; hd.res_pitch = d.res_pitch; hd.out = d.out; hd.out_pitch = d.out_pitch;
        hd.pool2 = c.pool;
        static HaloLaunch H;
        if (conv_halo_prepare(hd, num_sms, &H, err, sizeof(err))) { printf("[%s] halo prepare failed: %s\n", c.name, err); return 1; }
        if (conv_halo_launch(H, 0)) { printf("[%s] halo launch failed: %s\n", c.name, cudaGetErrorString(cudaGetLastError())); return 1; }
        L.grid = H.grid;
    } else {
    d.allow_split_k = 1;
    const bool want_strip = !strncmp(c.name, "strip", 5);
    options().strip = want_strip ? 2 : 1;  // "strip ..." cases force the strip form wherever it is legal
    const int prc = conv_tc_prepare(d, num_sms, c.block_n, &L, err, sizeof(err));
    options().strip = 1;
    if (prc) {
        printf("[%s] prepare failed: %s\n", c.name, err);
        return 1;
    }
    if (want_strip && !L.p.strip) printf("[%s] note: the strip form is not legal for this shape, im2col form checked\n", c.name);
    if (L.ws_bytes) {
        float* ws; int* cnt;
        CK(cudaMalloc(&ws, L.ws_bytes)); CK(cudaMalloc(&cnt, L.counter_ints * 4)); CK(cudaMemset(cnt, 0, L.counter_ints * 4));
        conv_tc_bind_workspace(&L, ws, cnt);
    }
    if (conv_tc_launch(L, 0)) {
        printf("[%s] launch failed: %s\n", c.name, cudaGetErrorString(cudaGetLastError()));
        return 1;
    }
    }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        printf("[%s] kernel failed: %s\n", c.name, cudaGetErrorString(e));
        exit(3);
    }
    std::vector<uint8_t> hout(out_bytes);
    CK(cudaMemcpy(hout.data(), dout, out_bytes, cudaMemcpyDeviceToHost));

    // CPU reference: the exact value and S = sum |x w| + |b| (+ |res|), held to the rounding model (see the file header)
    const bool halo_res = c.block_n == 2048 && c.residual;
    double max_err = 0, max_ref = 0, max_ratio = 0;
    long long bad = 0, first_bad_m = -1;
    int first_bad_n = -1;
    auto judge = [&](long long row, int co, double got, double bound, double v) {
        const double er = fabs(got - v);
        if (!(er <= bound)) {
            if (bad == 0) { first_bad_m = row; first_bad_n = co; }
            ++bad;
        }
        if (er > max_err || er != er) max_err = er;
        if (er / bound > max_ratio || er != er) max_ratio = er / bound;
        if (fabs(v) > max_ref) max_ref = fabs(v);
    };
    // fused pool: per window the maximum of the values, of |value| and of the summation term A
    const size_t npool = c.pool ? 1ULL * c.n * oh * ow * c.cout : 0;
    std::vector<double> pooled(npool, -1e300), pooled_abs(npool, 0.0), pooled_a(npool, 0.0);
    for (long long m = 0; m < M; ++m) {
        const int img = (int)(m / (ho * wo));
        const int rem = (int)(m % (ho * wo));
        const int oy = rem / wo, ox = rem % wo;
        for (int co = 0; co < c.cout; ++co) {
            double acc = 0, sabs = 0;
            for (int r = 0; r < c.k; ++r)
                for (int s = 0; s < c.k; ++s) {
                    const int iy = oy * c.stride - c.pad_lo + r, ix = ox * c.stride - c.pad_lo + s;
                    if (iy < 0 || iy >= c.h || ix < 0 || ix >= c.w) continue;
                    const float* xp = &x[((1LL * img * c.h + iy) * c.w + ix) * in_pitch];
                    const float* wp = &wt[1LL * co * K + (r * c.k + s) * c.cin];
                    for (int ci = 0; ci < c.cin; ++ci) {
                        const double p = double(xp[ci]) * wp[ci];
                        acc += p;
                        sabs += fabs(p);
                    }
                }
            double v = acc + bias[co], S = sabs + fabs(bias[co]);
            if (c.act) v = v > 0 ? v : v * double(0.1f);
            const double branch = v;
            if (c.residual) { v += res[m * c.cout + co]; S += fabs(res[m * c.cout + co]); }
            const double A = kU * (K + 4) * S;
            if (c.pool) {  // compared after the loop: maximum over the 2x2 window
                const size_t pi = ((1ULL * img * oh + oy / 2) * ow + ox / 2) * c.cout + co;
                if (v > pooled[pi]) pooled[pi] = v;
                pooled_abs[pi] = fmax(pooled_abs[pi], fabs(v));
                pooled_a[pi] = fmax(pooled_a[pi], A);
                continue;
            }
            const int ndst = c.upsample ? 4 : 1;
            for (int dd = 0; dd < ndst; ++dd) {
                long long row = m;
                if (c.upsample) row = (1LL * img * oh + 2 * oy + (dd >> 1)) * ow + 2 * ox + (dd & 1);
                float got;
                if (c.fp32) got = reinterpret_cast<float*>(hout.data())[row * out_pitch + co];
                else got = __bfloat162float(reinterpret_cast<__nv_bfloat16*>(hout.data())[row * out_pitch + co]);
                double bound = A;
                if (!c.fp32) bound += 0.5 * bf16_ulp(fmax(fabs(double(got)), fabs(v)));
                if (halo_res) bound += 0.5 * bf16_ulp(fabs(branch) + A);
                judge(m, co, got, bound, v);
            }
        }
    }
    for (size_t i = 0; i < pooled.size(); ++i) {
        const long long row = static_cast<long long>(i / c.cout);
        const int co = static_cast<int>(i % c.cout);
        const float got = __bfloat162float(reinterpret_cast<__nv_bfloat16*>(hout.data())[row * out_pitch + co]);
        judge(row, co, got, 0.5 * bf16_ulp(fmax(fabs(double(got)), pooled_abs[i] + pooled_a[i])) + pooled_a[i], pooled[i]);
    }
    // untouched padding channels of a bf16 slice must still hold the 0xFF fill
    long long clobbered = 0;
    if (!c.fp32) {
        const uint16_t* o = reinterpret_cast<const uint16_t*>(hout.data());
        for (long long row = 0; row < 1LL * c.n * oh * ow; ++row)
            for (int ch = c.cout; ch < out_pitch; ++ch)
                if (o[row * out_pitch + ch] != 0xFFFF) ++clobbered;
    }
    if (L.p.split_k > 1) {  // a second launch on the same workspace: the counters must have been left at zero
        CK(cudaMemset(dout, 0xFF, out_bytes));
        if (conv_tc_launch(L, 0) || cudaDeviceSynchronize() != cudaSuccess) { printf("[%s] relaunch failed\n", c.name); return 1; }
        std::vector<uint8_t> h2(out_bytes);
        CK(cudaMemcpy(h2.data(), dout, out_bytes, cudaMemcpyDeviceToHost));
        if (memcmp(h2.data(), hout.data(), out_bytes)) { printf("[%s] split-K relaunch differs\n", c.name); ++bad; }
    }
    printf("[%-28s] M=%lld N=%d K=%d bn=%d%s%s%s grid=%d  max_err=%.4g (max|ref|=%.3g, worst/bound=%.3f) bad=%lld clobbered=%lld %s\n",
           c.name, M, c.cout, K, L.block_n, L.two_cta ? (L.p.strip ? "x2 strip" : "x2") : "", L.p.swap ? "swap" : "", L.p.split_k > 1 ? " splitK" : "", L.grid, max_err, max_ref, max_ratio, bad, clobbered,
           (bad == 0 && clobbered == 0) ? "OK" : "FAIL");
    if (bad) printf("    first bad at m=%lld n=%d\n", first_bad_m, first_bad_n);
    cudaFree(dx); cudaFree(dw); cudaFree(dbias); cudaFree(dout);
    if (dr) cudaFree(dr);
    return (bad == 0 && clobbered == 0) ? 0 : 1;
}

static void time_case(const char* name, int n, int h, int cin, int cout, int k, int stride, int num_sms,
                      int block_n, int debug = 0, int residual = 0, int grid_limit = 0) {
    const int pad = k == 3 ? 1 : 0;
    ConvDesc d;
    memset(&d, 0, sizeof(d));
    const int ho = (h + 2 * pad - k) / stride + 1;
    const size_t in_e = 1ULL * n * h * h * cin, out_e = 1ULL * n * ho * ho * cout, w_e = 1ULL * cout * k * k * cin;
    __nv_bfloat16 *dx, *dw, *dout;
    float* dbias;
    CK(cudaMalloc(&dx, in_e * 2));
    CK(cudaMalloc(&dw, w_e * 2));
    CK(cudaMalloc(&dout, out_e * 2));
    CK(cudaMalloc(&dbias, 1024 * 4));
    CK(cudaMemset(dx, 0x3C, in_e * 2));  // bf16 0x3C3C ~ 0.0115
    CK(cudaMemset(dw, 0x3C, w_e * 2));
    CK(cudaMemset(dbias, 0, 1024 * 4));
    d.n = n; d.hi = h; d.wi = h; d.cin = cin; d.in_pitch = cin; d.in = dx;
    d.cout = cout; d.ksize = k; d.stride = stride; d.pad_lo = pad; d.pad_hi = pad;
    static float zero_bias[1024]; d.w = dw; d.bias = dbias; d.bias_host = zero_bias; d.act = 1; d.alpha = 0.1f;
    d.out = dout; d.out_pitch = cout;
    ConvLaunch L;
    char err[256] = {0};
    __nv_bfloat16* dres = nullptr;
    if (residual) { CK(cudaMalloc(&dres, out_e * 2)); CK(cudaMemset(dres, 0x3C, out_e * 2)); d.residual = dres; d.res_pitch = cout; }
    d.allow_split_k = getenv("FD_SPLITK") != nullptr;
    if (getenv("FD_STRIP")) options().strip = atoi(getenv("FD_STRIP"));  // harness only: 0 / 1 / 2
    if (conv_tc_prepare(d, num_sms, block_n, &L, err, sizeof(err))) { printf("[%s] prepare failed: %s\n", name, err); return; }
    if (L.ws_bytes) {
        float* ws; int* cnt;
        CK(cudaMalloc(&ws, L.ws_bytes)); CK(cudaMalloc(&cnt, L.counter_ints * 4)); CK(cudaMemset(cnt, 0, L.counter_ints * 4));
        conv_tc_bind_workspace(&L, ws, cnt);
        printf("    split_k = %d, workspace %.1f MB\n", L.p.split_k, L.ws_bytes / 1e6);
    }
    L.p.debug = debug;
    if (grid_limit && grid_limit < L.grid) L.grid = grid_limit;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int i = 0; i < 3; ++i) conv_tc_launch(L, 0);
    CK(cudaDeviceSynchronize());
    const int iters = 20;
    cudaEventRecord(e0);
    for (int i = 0; i < iters; ++i) conv_tc_launch(L, 0);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    ms /= iters;
    const double bytes = (in_e + out_e + w_e) * 2.0;
    if (getenv("FD_PROF")) {
        long long* dprof; CK(cudaMalloc(&dprof, 8 * 16 * 256)); CK(cudaMemset(dprof, 0, 8 * 16 * 256));
        L.p.prof = dprof;
        conv_tc_launch(L, 0); CK(cudaDeviceSynchronize());
        static long long hp[16 * 256]; CK(cudaMemcpy(hp, dprof, sizeof(hp), cudaMemcpyDeviceToHost));
        double a[16] = {0}, mx[16] = {0};
        for (int c = 0; c < L.grid; ++c) for (int q = 0; q < 16; ++q) { a[q] += double(hp[c * 16 + q]) / L.grid; if (hp[c * 16 + q] > mx[q]) mx[q] = double(hp[c * 16 + q]); }
        printf("    epilogue phases (avg cycles/CTA, group 0 warp 0): wait-acc %.0f | tmem-ld %.0f | res-fetch+bias loads %.0f | math %.0f | stage(STS+sync) %.0f | transposed read+stores %.0f\n", a[6], a[7], a[11], a[10], a[8], a[9]);
        printf("    prof max over CTAs: producer %.0f mma %.0f epi %.0f cycles; launch %.1f us -> %.0f cycles at 1.9 GHz\n", mx[0], mx[2], mx[5], ms * 1e3, ms * 1e-3 * 1.9e9);
        const double tiles_per_cta = double(L.p.num_m_tiles) * L.p.num_n_tiles / L.grid;
        printf("    prof(avg cycles/CTA, %.1f tiles x %d kb): producer total %.0f wait-empty %.0f | mma total %.0f wait-full %.0f wait-tmem %.0f | epi(g0) total %.0f wait-acc %.0f | per kb: %.0f cyc\n",
               tiles_per_cta, L.p.num_k_blocks, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[2] / (tiles_per_cta * L.p.num_k_blocks));
        L.p.prof = nullptr; cudaFree(dprof);
    }
    if (dres) cudaFree(dres);
    printf("[time %-24s dbg=%d res=%d grid=%3d] bn=%3d tiles=%6d  %.3f ms  %.1f TFLOP/s (%.2f per CTA)  %.0f GB/s(min traffic)\n", name, debug, residual, L.grid, L.block_n,
           L.p.num_m_tiles * L.p.num_n_tiles, ms, L.flops / ms * 1e-9, L.flops / ms * 1e-9 / L.grid, bytes / ms * 1e-6);
    cudaFree(dx); cudaFree(dw); cudaFree(dout); cudaFree(dbias);
}

int main(int argc, char** argv) {
    const char* mode = argc > 1 ? argv[1] : "all";
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("device: %s, %d SMs, cc %d.%d\n", prop.name, prop.multiProcessorCount, prop.major, prop.minor);
    char err[256] = {0};
    if (conv_tc_init(err, sizeof(err))) { printf("init failed: %s\n", err); return 2; }
    if (conv_halo_init()) { printf("conv_halo_init failed\n"); return 2; }
    const int sms = prop.multiProcessorCount;
    int fails = 0;
    if (!strcmp(mode, "check") || !strcmp(mode, "all")) {
        const Case cases[] = {
            // name                     n  h   w  cin cout k s pl ph act res fp32 up extra bn
            {"1x1 64->128",             2, 13, 13, 64, 128, 1, 1, 0, 0, 1, 0, 0, 0, 0, 0},
            {"1x1 64->128 pitch+64",    2, 13, 13, 64, 128, 1, 1, 0, 0, 1, 0, 0, 0, 64, 0},
            {"1x1 128->64 res",         1, 26, 26, 128, 64, 1, 1, 0, 0, 1, 1, 0, 0, 0, 0},
            {"1x1 256->255 head fp32",  2, 13, 13, 256, 255, 1, 1, 0, 0, 0, 0, 1, 0, 0, 0},
            {"1x1 128->42 head fp32",   1, 26, 26, 128, 42, 1, 1, 0, 0, 0, 0, 1, 0, 0, 0},
            {"1x1 256->128 upsample",   2, 13, 13, 256, 128, 1, 1, 0, 0, 1, 0, 0, 1, 0, 0},
            {"1x1 32->64 (bk32)",       1, 20, 20, 32, 64, 1, 1, 0, 0, 1, 0, 0, 0, 0, 0},
            {"3x3 64->64 s1",           2, 13, 13, 64, 64, 3, 1, 1, 1, 1, 0, 0, 0, 0, 0},
            {"3x3 64->128 s1 res",      3, 13, 13, 64, 128, 3, 1, 1, 1, 1, 1, 0, 0, 0, 0},
            {"3x3 64->128 s2",          2, 26, 26, 64, 128, 3, 2, 1, 1, 1, 0, 0, 0, 0, 0},
            {"3x3 64->128 s2 pad(1,0)", 2, 26, 26, 64, 128, 3, 2, 1, 0, 1, 0, 0, 0, 0, 0},
            {"3x3 32->64 s1 (bk32)",    2, 16, 16, 32, 64, 3, 1, 1, 1, 1, 0, 0, 0, 0, 0},
            {"3x3 32->64 s2 (bk32)",    1, 32, 32, 32, 64, 3, 2, 1, 1, 1, 0, 0, 0, 0, 0},
            {"3x3 128->512 s1 bn256",   2, 13, 13, 128, 512, 3, 1, 1, 1, 1, 0, 0, 0, 0, 256},
            {"3x3 128->512 s1 bn128",   2, 13, 13, 128, 512, 3, 1, 1, 1, 1, 0, 0, 0, 0, 128},
            {"3x3 64->32 pitch+32",     1, 19, 19, 64, 32, 3, 1, 1, 1, 1, 0, 0, 0, 32, 0},
            {"1x1 512->256 many tiles", 8, 26, 26, 512, 256, 1, 1, 0, 0, 1, 0, 0, 0, 0, 64},
            {"3x3 tiny map 64->64",     1, 5, 5, 64, 64, 3, 1, 1, 1, 1, 0, 0, 0, 0, 0},
            {"swap 3x3 64->128 res",    3, 13, 13, 64, 128, 3, 1, 1, 1, 1, 1, 0, 0, 0, 1024},
            {"swap 3x3 32->64 s2",      2, 32, 32, 32, 64, 3, 2, 1, 1, 1, 0, 0, 0, 0, 1024},
            {"swap 1x1 256->128 up",    2, 13, 13, 256, 128, 1, 1, 0, 0, 1, 0, 0, 1, 64, 1024},
            {"swap 1x1 64->32 pitch",   2, 20, 20, 64, 32, 1, 1, 0, 0, 1, 1, 0, 0, 64, 1024},
            {"swap 3x3 16->32 (bk16)",  2, 20, 20, 16, 32, 3, 1, 1, 1, 1, 0, 0, 0, 0, 1024},
            {"swap 1x1 384->128 big",   8, 52, 52, 384, 128, 1, 1, 0, 0, 1, 0, 0, 0, 0, 1024},
            {"2cta 3x3 128->512",       2, 13, 13, 128, 512, 3, 1, 1, 1, 1, 0, 0, 0, 0, 512},
            {"2cta 3x3 64->256 res s2", 3, 26, 26, 64, 256, 3, 2, 1, 1, 1, 1, 0, 0, 0, 512},
            {"2cta 1x1 256->255 fp32",  2, 13, 13, 256, 255, 1, 1, 0, 0, 0, 0, 1, 0, 0, 512},
            {"2cta 1x1 512->256 many",  8, 26, 26, 512, 256, 1, 1, 0, 0, 1, 1, 0, 0, 0, 512},
            {"2cta 1x1 256->256 up",    2, 13, 13, 256, 256, 1, 1, 0, 0, 1, 0, 0, 1, 64, 512},
            {"2cta 3x3 128->256 big",   16, 52, 52, 128, 256, 3, 1, 1, 1, 1, 1, 0, 0, 0, 512},
            // strip mode of the pair kernel (W >= 40): odd sizes, residual, two N tiles, the widest legal map (61: 256 strip rows)
            {"strip 3x3 64->256 odd",   3, 44, 41, 64, 256, 3, 1, 1, 1, 1, 1, 0, 0, 0, 512},
            {"strip 3x3 128->512 2n",   2, 52, 52, 128, 512, 3, 1, 1, 1, 1, 0, 0, 0, 64, 512},
            {"strip 3x3 64->256 w61",   1, 7, 61, 64, 256, 3, 1, 1, 1, 1, 1, 0, 0, 0, 512},
            {"strip 3x3 64->256 w62",   1, 7, 62, 64, 256, 3, 1, 1, 1, 1, 1, 0, 0, 0, 512},
            {"1cta 3x3 128->512",       2, 13, 13, 128, 512, 3, 1, 1, 1, 1, 0, 0, 0, 0, 257},
            // maps wider than 61 need strips of more than 256 positions (YOLOv3-608: 76x76), and the 608 grids 38 / 19
            {"strip 3x3 64->256 w76",   2, 9, 76, 64, 256, 3, 1, 1, 1, 1, 1, 0, 0, 0, 512},
            {"strip 3x3 128->256 76sq", 2, 76, 76, 128, 256, 3, 1, 1, 1, 1, 1, 0, 0, 0, 512},
            {"strip 3x3 64->512 38sq",  3, 38, 38, 64, 512, 3, 1, 1, 1, 1, 0, 0, 0, 0, 512},
            {"strip 3x3 64->256 19sq",  5, 19, 19, 64, 256, 3, 1, 1, 1, 1, 1, 0, 0, 0, 512},
            {"strip 3x3 128->256 13sq", 9, 13, 13, 128, 256, 3, 1, 1, 1, 1, 1, 0, 0, 0, 512},
            {"3x3 16->32 s1 (bk16)",    2, 20, 20, 16, 32, 3, 1, 1, 1, 1, 0, 0, 0, 0, 0},
            {"halo 3x3 32->64 s1 res",  2, 72, 76, 32, 64, 3, 1, 1, 1, 1, 1, 0, 0, 0, 2048},
            {"halo 3x3 32->64 s2",      2, 130, 134, 32, 64, 3, 2, 1, 1, 1, 0, 0, 0, 0, 2048},
            {"halo 3x3 32->32 s1 pitch",1, 64, 64, 32, 32, 3, 1, 1, 1, 0, 0, 0, 0, 32, 2048},
            {"halo 3x3 32->64 s2 (1,0)",1, 128, 128, 32, 64, 3, 2, 1, 0, 1, 0, 0, 0, 0, 2048},
            {"halo 3x3 16->32 s1",      2, 70, 66, 16, 32, 3, 1, 1, 1, 1, 0, 0, 0, 0, 2048},
            {"halo 3x3 64->128 s1 res", 2, 72, 68, 64, 128, 3, 1, 1, 1, 1, 1, 0, 0, 0, 2048},
            {"halo 3x3 64->64 s1",      1, 64, 64, 64, 64, 3, 1, 1, 1, 1, 0, 0, 0, 64, 2048},
            {"halo 3x3 16->64 s2 res",  1, 130, 128, 16, 64, 3, 2, 1, 1, 1, 1, 0, 0, 16, 2048},
            {"1x1 48->64 (bk16)",       1, 20, 20, 48, 64, 1, 1, 0, 0, 1, 0, 0, 0, 16, 0},
            // MaxPool(2, 2) fused into the halo-patch kernel's epilogue (YOLOv3-tiny: conv2 / conv3), incl. a map that is not a
            // multiple of the 16 x 8 tile and the rotating-buffer form (Cout 128)
            {"halo 3x3 16->32 pool",    2, 72, 68, 16, 32, 3, 1, 1, 1, 1, 0, 0, 0, 0, 2048, 1},
            {"halo 3x3 32->64 pool",    1, 104, 104, 32, 64, 3, 1, 1, 1, 1, 0, 0, 0, 0, 2048, 1},
            {"halo 3x3 64->128 pool",   1, 64, 66, 64, 128, 3, 1, 1, 1, 0, 0, 0, 0, 8, 2048, 1},
            // the production split-K shapes at batch 1 (13x13 3x3 512->1024 with and without a residual, 26x26 3x3 256->512)
            // and a split CTA-pair case forced with block_n 512
            {"splitK 3x3 512->1024 13sq",   1, 13, 13, 512, 1024, 3, 1, 1, 1, 1, 0, 0, 0, 0, 0},
            {"splitK 3x3 512->1024 13 res", 1, 13, 13, 512, 1024, 3, 1, 1, 1, 1, 1, 0, 0, 0, 0},
            {"splitK 3x3 256->512 26sq",    1, 26, 26, 256, 512, 3, 1, 1, 1, 1, 0, 0, 0, 0, 0},
            {"splitK 2cta 3x3 512->1024",   1, 13, 13, 512, 1024, 3, 1, 1, 1, 1, 1, 0, 0, 0, 512},
        };
        for (const Case& c : cases) fails += run_case(c, sms);
        printf("check: %d failing case(s)\n", fails);
    }
    if (!strcmp(mode, "alt")) {
        for (int dbg : {9, 73}) {
            time_case("3x3 32->64 s1 @208 bs64", 64, 208, 32, 64, 3, 1, sms, 0, dbg);
            time_case("3x3 64->128 @104 bs64", 64, 104, 64, 128, 3, 1, sms, 0, dbg);
            time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, 257, dbg);
        }
    }
    if (!strcmp(mode, "narrow")) {
        for (int dbg : {0, 1, 2, 4, 6, 7, 9}) time_case("3x3 32->64 s1 @208 bs64", 64, 208, 32, 64, 3, 1, sms, 0, dbg);
        for (int dbg : {0, 1, 9}) time_case("1x1 256->128 @52 bs64", 64, 52, 256, 128, 1, 1, sms, 0, dbg);
        for (int dbg : {0, 1, 9}) time_case("3x3 64->128 @104 bs64", 64, 104, 64, 128, 3, 1, sms, 0, dbg);
    }
    if (!strcmp(mode, "empty")) {
        for (int bn : {64, 128, 257, 512}) time_case("empty 1x1 512->256 @26", 64, 26, 512, 256, 1, 1, sms, bn, 32, 0);
        time_case("1 tile/CTA 1x1 512->256", 4, 26, 512, 256, 1, 1, sms, 257, 0, 0);
        time_case("1 tile/CTA 3x3 256->512", 28, 26, 256, 256, 3, 1, sms, 257, 0, 0);
    }
    if (!strcmp(mode, "one")) {
        for (int bn : {64, 128, 257, 512}) {
            time_case("1x1 512->256 @26 bs64", 64, 26, 512, 256, 1, 1, sms, bn, 0, 0);
            time_case("1x1 1024->512 @13 bs64", 64, 13, 1024, 512, 1, 1, sms, bn, 0, 0);
            time_case("1x1 256->128 @52 bs64", 64, 52, 256, 128, 1, 1, sms, bn > 128 ? 128 : bn, 0, 0);
            time_case("3x3 512->1024 @13 res", 64, 13, 512, 1024, 3, 1, sms, bn, 0, 1);
        }
    }
    if (!strcmp(mode, "mma")) {
        for (int bn : {257, 512})
            for (int dbg : {0, 1, 9, 25}) time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, bn, dbg);
        for (int dbg : {0, 9, 25}) time_case("3x3 64->128 @104 bs64", 64, 104, 64, 128, 3, 1, sms, 0, dbg);
        for (int dbg : {0, 9, 25}) time_case("3x3 32->64 s1 @208 bs64", 64, 208, 32, 64, 3, 1, sms, 0, dbg);
    }
    if (!strcmp(mode, "two")) {
        for (int bn : {257, 512}) {
            time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, bn);
            time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, bn, 0, 1);
            time_case("3x3 256->512 @26 bs64", 64, 26, 256, 512, 3, 1, sms, bn);
            time_case("3x3 512->1024 @13 bs64", 64, 13, 512, 1024, 3, 1, sms, bn);
            time_case("1x1 512->256 @26 bs64", 64, 26, 512, 256, 1, 1, sms, bn);
            time_case("1x1 1024->512 @13 bs64", 64, 13, 1024, 512, 1, 1, sms, bn);
            time_case("3x3 256->512 s2 @52 bs64", 64, 52, 256, 512, 3, 2, sms, bn);
        }
    }
    if (!strcmp(mode, "strip")) {  // run with FD_STRIP=0 / 1 / 2 to compare
        time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, 512);
        time_case("3x3 128->256 @52 bs64 res", 64, 52, 128, 256, 3, 1, sms, 512, 0, 1);
        time_case("3x3 256->512 @26 bs64", 64, 26, 256, 512, 3, 1, sms, 512);
        time_case("3x3 512->1024 @13 bs64", 64, 13, 512, 1024, 3, 1, sms, 512);
    }
    if (!strcmp(mode, "grid")) {
        for (int g : {148, 111, 74, 37, 16}) time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, 0, 0, 0, g);
        for (int g : {148, 74, 37}) time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, 0, 1, 0, g);
        for (int g : {148, 74, 37}) time_case("3x3 256->512 @26 bs64", 64, 26, 256, 512, 3, 1, sms, 0, 0, 0, g);
        for (int g : {148, 74, 37}) time_case("3x3 32->64 s1 @208 bs64", 64, 208, 32, 64, 3, 1, sms, 0, 0, 0, g);
        for (int g : {148, 74, 37}) time_case("3x3 32->64 s1 @208 bs64", 64, 208, 32, 64, 3, 1, sms, 0, 7, 0, g);
        for (int g : {148, 74, 37}) time_case("3x3 64->128 @104 bs64", 64, 104, 64, 128, 3, 1, sms, 0, 0, 0, g);
        for (int g : {148, 74, 37}) time_case("1x1 512->256 @26 bs64", 64, 26, 512, 256, 1, 1, sms, 0, 0, 0, g);
    }
    if (!strcmp(mode, "small")) {
        time_case("3x3 128->256 @52 bs1", 1, 52, 128, 256, 3, 1, sms, 0);
        time_case("3x3 256->512 @26 bs1", 1, 26, 256, 512, 3, 1, sms, 0);
        time_case("3x3 512->1024 @13 bs1", 1, 13, 512, 1024, 3, 1, sms, 0);
        time_case("1x1 1024->512 @13 bs1", 1, 13, 1024, 512, 1, 1, sms, 0);
        time_case("3x3 512->1024 @13 bs8", 8, 13, 512, 1024, 3, 1, sms, 0);
    }
    if (!strcmp(mode, "epi")) {
        for (int dbg : {0, 1, 2, 4, 6, 8}) time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, 0, dbg);
        for (int dbg : {0, 1, 2, 4, 6}) time_case("1x1 512->256 @26 bs64", 64, 26, 512, 256, 1, 1, sms, 0, dbg);
        for (int dbg : {0, 4}) time_case("1x1 256->128 @52 bs64", 64, 52, 256, 128, 1, 1, sms, 0, dbg);
    }
    if (!strcmp(mode, "probe")) {
        for (int dbg : {0, 1, 2, 4, 3, 5, 6, 7}) time_case("3x3 32->64 s2 @416 bs64", 64, 416, 32, 64, 3, 2, sms, 0, dbg);
        for (int dbg : {0, 1, 2, 4}) time_case("3x3 32->64 s1 @208 bs64", 64, 208, 32, 64, 3, 1, sms, 0, dbg);
        for (int dbg : {0, 1, 2, 4}) time_case("3x3 64->128 @104 bs64", 64, 104, 64, 128, 3, 1, sms, 0, dbg);
        for (int dbg : {0, 1, 2, 4}) time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, 0, dbg);
        for (int dbg : {0, 1}) time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, 0, dbg, 1);
        for (int dbg : {0, 1, 2, 4}) time_case("1x1 1024->512 @13 bs64", 64, 13, 1024, 512, 1, 1, sms, 0, dbg);
        for (int dbg : {0, 1, 2, 4}) time_case("1x1 64->32 @208 bs64", 64, 208, 64, 32, 1, 1, sms, 0, dbg);
    }
    if (!strcmp(mode, "time") || !strcmp(mode, "all")) {
        time_case("3x3 128->256 @52 bs64", 64, 52, 128, 256, 3, 1, sms, 0);
        time_case("3x3 256->512 @26 bs64", 64, 26, 256, 512, 3, 1, sms, 0);
        time_case("3x3 256->512 @26 bn128", 64, 26, 256, 512, 3, 1, sms, 128);
        time_case("3x3 512->1024 @13 bs64", 64, 13, 512, 1024, 3, 1, sms, 0);
        time_case("3x3 512->1024 @13 bn128", 64, 13, 512, 1024, 3, 1, sms, 128);
        time_case("1x1 256->128 @52 bs64", 64, 52, 256, 128, 1, 1, sms, 0);
        time_case("1x1 512->256 @26 bs64", 64, 26, 512, 256, 1, 1, sms, 0);
        time_case("1x1 1024->512 @13 bs64", 64, 13, 1024, 512, 1, 1, sms, 0);
        time_case("3x3 64->128 @104 bs64", 64, 104, 64, 128, 3, 1, sms, 0);
        time_case("3x3 32->64 s2 @416 bs64", 64, 416, 32, 64, 3, 2, sms, 0);
        time_case("3x3 512->1024 @13 bs1", 1, 13, 512, 1024, 3, 1, sms, 0);
    }
    return fails ? 1 : 0;
}
