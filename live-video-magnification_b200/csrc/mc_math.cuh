// Per-pixel arithmetic shared by the kernels.  Everything here is __host__ __device__ so the CPU
// test-suite can compile the *same* functions into a check library (tests/hostcheck) and compare
// them with the oracle without a GPU; the product never calls them on the host.
#pragma once
#include <cstdint>
#include <cmath>

#if defined(__CUDACC__)
#define MC_HD __host__ __device__ __forceinline__
#else
#define MC_HD inline
#endif

namespace mc {

constexpr int kLabLutDim = 33;          // OpenCV LAB_LUT_DIM
constexpr int kGammaTabSize = 1024;     // OpenCV GAMMA_TAB_SIZE

// One packed LUT cell (32 B = one L1/L2 sector): the Lab int16 values of the lattice points (b, g..g+1, r..r+1),
// interleaved so that one dp2a does the r-interpolation of a channel at one (b, g) corner.  A pixel needs two cells,
// (b, g, r) and (b+1, g, r), each fetched with ONE 256-bit load (LDG.E.256 on sm_100) — the divergent LUT gathers are
// what bounds the BGR->Lab kernels (L1 tag lookups per distinct sector), so bytes per gather instruction is the lever.
// The table is [34][33][33]: g+1 / r+1 are clamped when the table is built and the b = 33 slab repeats b = 32, so the
// device code needs no clamping (a clamped neighbour always has weight 0).
struct alignas(32) LabLutCell { int16_t v[16]; };  // {L00,L01, a00,a01, b00,b01, L10,L11, a10,a11, b10,b11, 0,0,0,0}, index = (g-offset, r-offset)
constexpr int kLabLutSlab = kLabLutDim * kLabLutDim;   // cells per b slab
constexpr int kLabLutCells = (kLabLutDim + 1) * kLabLutSlab;

MC_HD int reflect101(int i, int n) {
    if (i < 0) i = -i;
    if (i >= n) i = 2 * n - 2 - i;
    return i < 0 ? 0 : (i >= n ? n - 1 : i);
}

// pyrUp source-index rule (cv::pyrUp, SURVEY A.2): s[-1] := s[1], s[n] := s[n-1].
MC_HD int upsrc(int i, int n) {
    if (i < 0) return 1;
    if (i >= n) return n - 1;
    return i;
}

// u8 -> f32 as Mat::convertTo(CV_32F, 1/255) does it (MagnifyCore.hpp:89): x * (float)(1/255).
MC_HD float u8_to_unit(uint8_t v) { return (float)v * 0.003921568859368563f; }

// f32 -> u8 as Mat::convertTo(CV_8U, 255, 1/255) does it (MagnifyCore.hpp:153):
// saturate(round_half_even(fma(x, 255, (float)(1/255)))).
// OpenCV rounds with cvtps2dq: NaN and anything outside the int32 range become INT_MIN and then saturate to 0.
MC_HD uint8_t unit_to_u8(float x) {
    float v = fmaf(x, 255.0f, 0.003921568859368563f);
    v = rintf(v);
    if (!(v > 0.0f) || v >= 2147483648.0f) return 0;   // NaN, negatives, +inf / out of int range -> 0
    if (v > 255.0f) return 255;
    return (uint8_t)(int)v;
}

// same on the device in one conversion instruction: cvt.rni.u8.f32 rounds half to even and clamps to [0, 255]
// (float -> integer conversions saturate; NaN -> 0), which is exactly cvRound + saturate_cast<uchar>.
MC_HD uint8_t unit01_to_u8(float x) {
#if defined(__CUDA_ARCH__) && !defined(MC_CUDA_EMU)
    unsigned r;
    asm("cvt.rni.u8.f32 %0, %1;" : "=r"(r) : "f"(fmaf(x, 255.0f, 0.003921568859368563f)));
    return (uint8_t)r;
#else
    return unit_to_u8(x);
#endif
}

// generic convertTo(CV_8U, alpha, beta) used by Color egress (MagnifyCore.hpp:202-203)
MC_HD uint8_t scaled_to_u8(float x, float a, float b) {
    float v = rintf(fmaf(x, a, b));
    if (!(v > 0.0f) || v >= 2147483648.0f) return 0;   // as unit_to_u8: cvtps2dq semantics
    if (v > 255.0f) return 255;
    return (uint8_t)(int)v;
}

#if defined(__CUDACC__)
#define MC_LDG16(p) __ldg(reinterpret_cast<const int4*>(p))
#endif

// Per-channel quantisation of a u8 sample as OpenCV's float path sees it: cx = cvRound(v*(1/255)*2^14),
// LUT cell t = cx >> 9 and 4-bit weight x = (cx >> 5) & 15.  Returned packed as q = cx >> 5 = (t << 4) | x.
// cx equals (v*16448 + 128) >> 8 for all 256 inputs (tests/test_host.py checks it against the float form), so the
// kernels compute q with one IMAD and a shift instead of a table lookup.
MC_HD int lab_q_of_u8_float(int v) {   // the definition (float arithmetic of convertTo + cvtColor)
    const float c = ((float)v * 0.003921568859368563f) * 16384.0f;
#if defined(__CUDA_ARCH__)
    const int cx = __float2int_rn(c);
#else
    const int cx = (int)lrintf(c);
#endif
    return cx >> 5;
}
MC_HD int lab_q_of_u8(int v) { return (v * 16448 + 128) >> 13; }

#if defined(__CUDA_ARCH__)
// one LUT cell = one 256-bit read-only load
__device__ __forceinline__ void ldg_cell(const LabLutCell* p, int (&w)[8]) {
#if defined(MC_CUDA_EMU)
    const int* q = reinterpret_cast<const int*>(p);
    for (int i = 0; i < 8; ++i) w[i] = q[i];
#else
    asm("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "l"(p));
#endif
}
#endif

// cv::cvtColor(COLOR_BGR2Lab) on CV_32F input that came from u8/255 — bit-exact restatement of
// OpenCV's 33^3 int16 LUT + 4-bit fixed-point trilinear interpolation (SURVEY.md A.3).
// qb/qg/qr are lab_q_of_u8() of the three samples.  Fixed-point result: L*2^14/100, (a+128)*64, (b+128)*64.
MC_HD void lab_fixed_from_q(int qb, int qg, int qr, const LabLutCell* __restrict__ lut, int& sL, int& sA, int& sB) {
    const int tb = qb >> 4, tg = qg >> 4, tr = qr >> 4;
    const int xb = qb & 15, xg = qg & 15, xr = qr & 15;
    const LabLutCell* c0 = lut + ((tb * kLabLutDim + tg) * kLabLutDim + tr);
    const int w01 = (16 - xb) * xg, w00 = ((16 - xb) << 4) - w01, w11 = xb * xg, w10 = (xb << 4) - w11;
#if defined(__CUDA_ARCH__)
    int u[8], v[8];
    ldg_cell(c0, u);
    ldg_cell(c0 + kLabLutSlab, v);
    const int wr = 16 + 255 * xr;                               // int8 pair for dp2a: lo * (16-x) + hi * x
    sL = w00 * __dp2a_lo(u[0], wr, 0) + (w01 * __dp2a_lo(u[3], wr, 0) + (w10 * __dp2a_lo(v[0], wr, 0) + (w11 * __dp2a_lo(v[3], wr, 0) + 2048)));
    sA = w00 * __dp2a_lo(u[1], wr, 0) + (w01 * __dp2a_lo(u[4], wr, 0) + (w10 * __dp2a_lo(v[1], wr, 0) + (w11 * __dp2a_lo(v[4], wr, 0) + 2048)));
    sB = w00 * __dp2a_lo(u[2], wr, 0) + (w01 * __dp2a_lo(u[5], wr, 0) + (w10 * __dp2a_lo(v[2], wr, 0) + (w11 * __dp2a_lo(v[5], wr, 0) + 2048)));
#else
    const LabLutCell* cs[2] = {c0, c0 + kLabLutSlab};
    const int ws[2][2] = {{w00, w01}, {w10, w11}};
    sL = sA = sB = 2048;
    for (int ib = 0; ib < 2; ++ib)
        for (int ig = 0; ig < 2; ++ig) {
            const int16_t* e = cs[ib]->v + 6 * ig;
            sL += ws[ib][ig] * ((16 - xr) * e[0] + xr * e[1]);
            sA += ws[ib][ig] * ((16 - xr) * e[2] + xr * e[3]);
            sB += ws[ib][ig] * ((16 - xr) * e[4] + xr * e[5]);
        }
#endif
    sL >>= 12;
    sA >>= 12;
    sB >>= 12;
}

MC_HD void bgr_u8_to_lab_fixed(uint8_t b8, uint8_t g8, uint8_t r8, const LabLutCell* __restrict__ lut,
                               int& sL, int& sA, int& sB) {
    lab_fixed_from_q(lab_q_of_u8(b8), lab_q_of_u8(g8), lab_q_of_u8(r8), lut, sL, sA, sB);
}

// Float Lab as OpenCV returns it: L in [0,100], a,b in [-128,128).
MC_HD void bgr_u8_to_lab(uint8_t b8, uint8_t g8, uint8_t r8, const LabLutCell* __restrict__ lut,
                         float& L, float& A, float& B) {
    int sL, sA, sB;
    bgr_u8_to_lab_fixed(b8, g8, r8, lut, sL, sA, sB);
    L = (float)sL * (100.0f / 16384.0f);
    A = fmaf((float)sA, 1.0f / 64.0f, -128.0f);
    B = fmaf((float)sB, 1.0f / 64.0f, -128.0f);
}

// Coefficients for Lab -> BGR (XYZ2sRGB_D65 rows scaled by the D65 white point), filled on the host.
struct LabInvCoeffs { float c[9]; };  // rows: B, G, R ; columns: X, Y, Z

MC_HD float spline_gamma(float v, const float4* __restrict__ tab) {
    // OpenCV splineInterpolate(x*GAMMA_TAB_SIZE, sRGBInvGammaTab, GAMMA_TAB_SIZE)
    const float xs = v * (float)kGammaTabSize;
    int ix = (int)xs;
    ix = ix < 0 ? 0 : (ix > kGammaTabSize - 1 ? kGammaTabSize - 1 : ix);
    const float fr = xs - (float)ix;
#if defined(__CUDA_ARCH__)
    const float4 t = __ldg(tab + ix);
#else
    const float4 t = tab[ix];
#endif
    return ((t.w * fr + t.z) * fr + t.y) * fr + t.x;
}

// Inverse sRGB transfer as OpenCV evaluates it.  OpenCV's 1024-segment spline only departs from the
// analytic curve in its first 8 segments (up to 7.8e-5 at the knee v = 0.0031; < 2e-7 for v >= 8/1024), so
// there the device evaluates 1.055 v^(1/2.4) - 0.055 with two SFU ops instead of a table gather, and keeps the
// spline itself for the dark end where the difference matters.
MC_HD float inv_gamma(float v, const float4* __restrict__ tab) {
#if defined(__CUDA_ARCH__)
    if (v >= 8.0f / 1024.0f) return fmaf(1.055f, exp2f(__log2f(v) * (1.0f / 2.4f)), -0.055f);
#endif
    return spline_gamma(v, tab);
}

// cv::cvtColor(COLOR_Lab2BGR) on CV_32F (analytic inverse + spline-interpolated sRGB gamma,
// output clipped to [0,1]); restated from OpenCV's Lab2RGBfloat, checked against cv2 to ~1e-5.
MC_HD void lab_to_bgr(float L, float a, float b, const LabInvCoeffs& k, const float4* __restrict__ gtab,
                      float& ob, float& og, float& orr) {
    // constant divisions are written as reciprocal multiplies (<= 1 ulp from the divide; the parity
    // budget is 1e-4) — IEEE divides would triple the instruction count of the egress kernel
    float Y, fy;
    if (L <= 8.0f) {
        Y = L * (1.0f / 903.3f);
        fy = 7.787f * Y + 16.0f / 116.0f;
    } else {
        fy = (L + 16.0f) * (1.0f / 116.0f);
        Y = fy * fy * fy;
    }
    float fx = a * (1.0f / 500.0f) + fy;
    float fz = fy - b * (1.0f / 200.0f);
    const float fth = 6.0f / 29.0f;
    const float X = fx <= fth ? (fx - 16.0f / 116.0f) * (1.0f / 7.787f) : fx * fx * fx;
    const float Z = fz <= fth ? (fz - 16.0f / 116.0f) * (1.0f / 7.787f) : fz * fz * fz;
    float vb = k.c[0] * X + k.c[1] * Y + k.c[2] * Z;
    float vg = k.c[3] * X + k.c[4] * Y + k.c[5] * Z;
    float vr = k.c[6] * X + k.c[7] * Y + k.c[8] * Z;
    // OpenCV clips as max(min(v, 1), 0) with SSE operand rules, so a NaN (Riesz: 0/0 in flat regions, SURVEY A.6-9)
    // comes out as 1.0 — white — not 0; fminf/fmaxf return the non-NaN operand, which gives exactly that
    vb = fmaxf(fminf(vb, 1.0f), 0.0f);
    vg = fmaxf(fminf(vg, 1.0f), 0.0f);
    vr = fmaxf(fminf(vr, 1.0f), 0.0f);
    ob = inv_gamma(vb, gtab);
    og = inv_gamma(vg, gtab);
    orr = inv_gamma(vr, gtab);
}

#if defined(__CUDACC__)
// Device-only, branch-lean form of lab_to_bgr for the egress kernels: identical arithmetic for the XYZ part
// (selects instead of branches), the [0,1] clip folded into saturating adds, and the gamma evaluated as
// 1.055 * 2^(log2(v)/2.4) - 0.055 with lg2/ex2.approx.ftz; only when one of the three linear values is below
// 8/1024 (where OpenCV's spline departs from the analytic curve) is the spline table consulted.
#if defined(MC_CUDA_EMU)   // CPU logic emulation for GPU-less CI (tests/cuda_emu): libm instead of the SFU
__device__ __forceinline__ float mc_lg2(float x) { return log2f(x); }
__device__ __forceinline__ float mc_ex2(float x) { return exp2f(x); }
#else
__device__ __forceinline__ float mc_lg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float mc_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
#endif

// NAN_AS_OPENCV: clip as OpenCV does (max(min(v, 1), 0): NaN -> 1.0, white).  Phase (Riesz) needs it — its L plane is
// NaN wherever the blurred amplitude is 0, e.g. in letterbox bars — Motion (Laplace) cannot produce a NaN and keeps
// the clip folded into the FFMA (.SAT, NaN -> 0) of its issue-bound egress kernel.
// G_R_FROM_Y: which product of the XYZ -> BGR dot products is rounded on its own (the other two are fused onto it, X
// before Z, or Y before Z): X for all three rows, or X for b and Y for g and r.  The rounding is pinned with intrinsics
// so that every instantiation of one kernel gives the same bits whatever code surrounds it (left to the compiler, the
// choice followed the surrounding code); the Motion egress kernels use the second form, the Phase egress the first.
template <bool NAN_AS_OPENCV = false, bool G_R_FROM_Y = false>
__device__ __forceinline__ void lab_to_bgr_fast(float L, float a, float b, const LabInvCoeffs& k,
                                                const float4* __restrict__ gtab, float& ob, float& og, float& orr) {
    const float y_lin = L * (1.0f / 903.3f);
    const float fy_lin = 7.787f * y_lin + 16.0f / 116.0f;
    const float fy_cub = (L + 16.0f) * (1.0f / 116.0f);
    const bool lo = L <= 8.0f;
    const float fy = lo ? fy_lin : fy_cub;
    const float Y = lo ? y_lin : fy_cub * fy_cub * fy_cub;
    const float fx = a * (1.0f / 500.0f) + fy;
    const float fz = fy - b * (1.0f / 200.0f);
    const float fth = 6.0f / 29.0f;
    const float X = fx <= fth ? (fx - 16.0f / 116.0f) * (1.0f / 7.787f) : fx * fx * fx;
    const float Z = fz <= fth ? (fz - 16.0f / 116.0f) * (1.0f / 7.787f) : fz * fz * fz;
    float vb = __fmaf_rn(k.c[2], Z, __fmaf_rn(k.c[1], Y, __fmul_rn(k.c[0], X)));
    float vg = G_R_FROM_Y ? __fmaf_rn(k.c[5], Z, __fmaf_rn(k.c[3], X, __fmul_rn(k.c[4], Y)))
                          : __fmaf_rn(k.c[5], Z, __fmaf_rn(k.c[4], Y, __fmul_rn(k.c[3], X)));
    float vr = G_R_FROM_Y ? __fmaf_rn(k.c[8], Z, __fmaf_rn(k.c[6], X, __fmul_rn(k.c[7], Y)))
                          : __fmaf_rn(k.c[8], Z, __fmaf_rn(k.c[7], Y, __fmul_rn(k.c[6], X)));
    if (NAN_AS_OPENCV) {
        // NOT fmaxf(fminf(v, 1), 0): ptxas folds that pair into the producing FFMA as .SAT, and .SAT turns NaN into 0
        // (black) where OpenCV's max(min(v,1),0) gives 1 (white).  The explicit NaN select survives the fold
        // (round-1 GPUTEST failure; tools/check_sass.py asserts the FSETP.NAN/FSEL pair is in k_riesz_egress).
        vb = (vb != vb) ? 1.0f : __saturatef(vb);
        vg = (vg != vg) ? 1.0f : __saturatef(vg);
        vr = (vr != vr) ? 1.0f : __saturatef(vr);
    } else {
        vb = __saturatef(vb); vg = __saturatef(vg); vr = __saturatef(vr);
    }
    ob = fmaf(1.055f, mc_ex2(mc_lg2(vb) * (1.0f / 2.4f)), -0.055f);
    og = fmaf(1.055f, mc_ex2(mc_lg2(vg) * (1.0f / 2.4f)), -0.055f);
    orr = fmaf(1.055f, mc_ex2(mc_lg2(vr) * (1.0f / 2.4f)), -0.055f);
    if (fminf(vb, fminf(vg, vr)) < 8.0f / 1024.0f) {   // dark end: OpenCV's spline, per channel
        if (vb < 8.0f / 1024.0f) ob = spline_gamma(vb, gtab);
        if (vg < 8.0f / 1024.0f) og = spline_gamma(vg, gtab);
        if (vr < 8.0f / 1024.0f) orr = spline_gamma(vr, gtab);
    }
}
#endif

// ------------------------------------------------------------------------------------------------
// Front of the reference chain (SURVEY.md 8f-1): GrayscaleProcessor and PreprocessProcessor arithmetic,
// restated from OpenCV's u8 paths and checked bit-exact against cv2 on the CPU (tests/test_host.py).
// ------------------------------------------------------------------------------------------------
// cv::cvtColor(COLOR_BGR2GRAY) on u8 (GrayscaleProcessor.cpp:13): 15-bit fixed point, round to nearest.
MC_HD uint8_t bgr_to_gray_u8(int b, int g, int r) { return (uint8_t)((b * 3735 + g * 19235 + r * 9798 + 16384) >> 15); }

#if defined(__CUDA_ARCH__)
#define MC_FMUL(a, b) __fmul_rn((a), (b))
#define MC_FADD(a, b) __fadd_rn((a), (b))
#define MC_RINT_I(x) __float2int_rn(x)
#else
#define MC_FMUL(a, b) ((a) * (b))      // host build uses -ffp-contract=off
#define MC_FADD(a, b) ((a) + (b))
#define MC_RINT_I(x) ((int)lrintf(x))
#endif

struct AreaTap { int di, si; float alpha; };   // OpenCV's DecimateAlpha: destination index, source index, weight

// cv::resize(INTER_AREA) for u8 (PreprocessProcessor.cpp:42), one output sample (dy, dx, channel ch).
//  * integer scale on both axes ("area fast"): 2x2 -> (sum + 2) >> 2 ; otherwise rint(int_sum * (1.f / area))
//  * otherwise: per contributing source row a float row sum  buf = sum_k S * alpha_k  (sequential, no FMA),
//    accumulated over rows as  sum = beta * buf  /  sum += beta * buf ; result rint(sum), saturated.
// xtab / ytab list the taps grouped by destination index; xofs[dx] .. xofs[dx+1] are dx's taps.
MC_HD uint8_t resize_area_sample(const uint8_t* __restrict__ src, size_t step, int cn, int ch, int dy, int dx,
                                 int iscale_x, int iscale_y, bool area_fast, const AreaTap* __restrict__ xtab,
                                 const int* __restrict__ xofs, const AreaTap* __restrict__ ytab,
                                 const int* __restrict__ yofs) {
    if (area_fast) {
        int sum = 0;
        for (int sy = 0; sy < iscale_y; ++sy) {
            const uint8_t* row = src + (size_t)(dy * iscale_y + sy) * step + (size_t)(dx * iscale_x) * cn + ch;
            for (int sx = 0; sx < iscale_x; ++sx) sum += row[(size_t)sx * cn];
        }
        if (iscale_x == 2 && iscale_y == 2) return (uint8_t)((sum + 2) >> 2);
        const float scale = 1.f / (float)(iscale_x * iscale_y);
        int v = MC_RINT_I(MC_FMUL((float)sum, scale));
        return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
    }
    float sum = 0.f;
    bool first = true;
    for (int j = yofs[dy]; j < yofs[dy + 1]; ++j) {
        const uint8_t* row = src + (size_t)ytab[j].si * step + ch;
        float buf = 0.f;
        for (int k = xofs[dx]; k < xofs[dx + 1]; ++k) buf = MC_FADD(buf, MC_FMUL((float)row[(size_t)xtab[k].si * cn], xtab[k].alpha));
        const float t = MC_FMUL(ytab[j].alpha, buf);
        sum = first ? t : MC_FADD(sum, t);
        first = false;
    }
    int v = MC_RINT_I(sum);
    return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// iirFilter (TemporalFilter.cpp:9-22): cv::addWeighted rounds once from a double sum (SURVEY A.5).
MC_HD float ema(float state, float x, double one_minus_c, double c) {
    return (float)((double)state * one_minus_c + (double)x * c);
}

}  // namespace mc
