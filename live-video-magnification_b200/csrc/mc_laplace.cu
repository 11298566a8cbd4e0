// Motion (Laplace) kernels for sm_100a.
//
//   lab16   : u8 BGR -> Lab (OpenCV LUT, exact) stored as int16 planes            (MagnifyCore.hpp:87-93)
//   level   : pyrDown + pyrUp + subtract + dual-EMA state update + gain, fused    (SpatialFilter.cpp:25-38,
//             per pyramid level; input f32 planes, Lab16 planes or u8 gray        TemporalFilter.cpp:9-22, MagnifyCore.hpp:127-134)
//   collapse: pyrUp + add (small levels only)                                     (SpatialFilter.cpp:52-61)
//   egress  : two pyrUp+add levels + chroma attenuation + input+motion +          (MagnifyCore.hpp:136-158)
//             Lab2BGR + u8
//
// All are bandwidth-bound stencil / pointwise kernels (no tensor cores).  Each CTA stages one tile
// (+halo) in shared memory with 128-bit loads, runs the separable 5-tap passes out of that tile, and
// each thread owns a 4x2 pixel block so state planes move as 128-bit coalesced vectors.  Tiles that
// touch an image border take a generic (slower) path that applies OpenCV's border rules.
#include <cuda.h>   // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint)

#include "mc_internal.h"
#include "mc_tma.cuh"

namespace mc {

namespace {

// request a line into L1 ahead of its use (no register is tied up, unlike a load issued early)
__device__ __forceinline__ void prefetch_l1(const void* p) {
#if !defined(MC_CUDA_EMU)
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
#else
    (void)p;
#endif
}

constexpr float kInv256 = 1.0f / 256.0f;
constexpr float kInv64 = 1.0f / 64.0f;

__device__ __forceinline__ float down5(float a, float b, float c, float d, float e) {
    // cv::pyrDown row/column pass: c*6 + (b+d)*4 + a + e
    return c * 6.0f + (b + d) * 4.0f + a + e;
}

// cv::pyrUp taps of the synthesis kernels (collapse, both egress forms).  The rounding is pinned with intrinsics — the
// 6-tap term as one FMA, which is what nvcc contracts it to anyway — so that every kernel evaluating the same tap gives
// the same bits whatever the surrounding code looks like (the strip and tile egress kernels are tested bit-identical).
__device__ __forceinline__ float up3(float a, float b, float c) { return __fadd_rn(__fmaf_rn(b, 6.0f, a), c); }   // a + 6 b + c
__device__ __forceinline__ float up2(float a, float b) { return __fmul_rn(__fadd_rn(a, b), 4.0f); }               // (a + b) * 4
__device__ __forceinline__ float band_of(float hi, float lo, float gain) { return __fmul_rn(__fsub_rn(hi, lo), gain); }

// ------------------------------------------------------------------------------------------------
// lab16: pointwise, 4 pixels per thread (12 input bytes = three 32-bit words).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_lab16(const uint8_t* __restrict__ in, size_t in_step, size_t in_lane_stride,
                                               int w, int h, const LabLutCell* __restrict__ lut,
                                               int16_t* __restrict__ lab, int pitch16, size_t plane16, int aligned,
                                               float* __restrict__ lf, int lf_pitch, size_t lf_plane) {
    const int lane = blockIdx.z;
    const int y = blockIdx.y;
    const int x = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (x >= w) return;
    const uint8_t* p = in + (size_t)lane * in_lane_stride + (size_t)y * in_step + (size_t)x * 3;
    uint8_t px[12];
    if (aligned && x + 4 <= w) {
        const uint32_t* q = reinterpret_cast<const uint32_t*>(p);
        const uint32_t a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            px[i] = (a >> (8 * i)) & 0xff;
            px[4 + i] = (b >> (8 * i)) & 0xff;
            px[8 + i] = (c >> (8 * i)) & 0xff;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 12; ++i) px[i] = (x + i / 3 < w) ? __ldg(p + i) : 0;
    }
    short L[4], A[4], B[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int sL, sA, sB;
        lab_fixed_from_q(lab_q_of_u8(px[3 * i]), lab_q_of_u8(px[3 * i + 1]), lab_q_of_u8(px[3 * i + 2]), lut, sL, sA, sB);
        L[i] = (short)sL; A[i] = (short)sA; B[i] = (short)sB;
    }
    int16_t* o = lab + (size_t)(lane * 3) * plane16 + (size_t)y * pitch16 + x;  // pitch16 % 64 == 0, x % 4 == 0
    *reinterpret_cast<short4*>(o) = make_short4(L[0], L[1], L[2], L[3]);
    *reinterpret_cast<short4*>(o + plane16) = make_short4(A[0], A[1], A[2], A[3]);
    *reinterpret_cast<short4*>(o + 2 * plane16) = make_short4(B[0], B[1], B[2], B[3]);
    if (lf) {   // Phase magnifies the L plane only (MagnifyCore.hpp:217-222): emit it as f32 too (rows padded to 32 floats)
        const float k = 100.0f / 16384.0f;
        *reinterpret_cast<float4*>(lf + (size_t)lane * lf_plane + (size_t)y * lf_pitch + x) =
            make_float4((float)L[0] * k, (float)L[1] * k, (float)L[2] * k, (float)L[3] * k);
    }
}

// ------------------------------------------------------------------------------------------------
// level: tile = 64 x 32 fine pixels, 256 threads, thread block of 4 x 2 pixels.
// ------------------------------------------------------------------------------------------------
constexpr int TW = 64, TH = 32;
constexpr int GW = TW + 8, GH = TH + 7;       // fine window 72 (71 used) x 39, origin (x0-4, y0-4)
constexpr int DW = TW / 2 + 2, DH = TH / 2 + 2;  // coarse window 34 x 18, origin (x0/2-1, y0/2-1)
constexpr int DP = 36;                        // coarse window pitch (8-byte aligned rows)

enum { IN_F32 = 0, IN_LAB16 = 1, IN_U8 = 2 };

template <int KIND>
__device__ __forceinline__ float load_scalar(const void* base, size_t off, float sc, float of) {
    if (KIND == IN_F32) return __ldg(reinterpret_cast<const float*>(base) + off);
    if (KIND == IN_LAB16) return fmaf((float)__ldg(reinterpret_cast<const short*>(base) + off), sc, of);
    return (float)__ldg(reinterpret_cast<const uint8_t*>(base) + off) * sc;
}

// Loads the fine window (GH x GW) of one plane into sG.  Interior tiles: 128-bit (or 64/32-bit for
// narrow element types) vector loads; border tiles: scalar loads with BORDER_REFLECT_101.
template <int KIND>
__device__ __forceinline__ void load_fine_window(float (*sG)[GW], const void* base, int row_stride, int wf, int hf,
                                                 int x0, int y0, bool interior, float sc, float of) {
    if (interior) {
        for (int i = threadIdx.x; i < GH * (GW / 4); i += 256) {
            const int r = i / (GW / 4), c4 = i - r * (GW / 4);
            const size_t off = (size_t)(y0 - 4 + r) * row_stride + (x0 - 4 + 4 * c4);
            float4 v;
            if (KIND == IN_F32) {
                v = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + off));
            } else if (KIND == IN_LAB16) {
                const short4 s = __ldg(reinterpret_cast<const short4*>(reinterpret_cast<const short*>(base) + off));
                v = make_float4(fmaf((float)s.x, sc, of), fmaf((float)s.y, sc, of), fmaf((float)s.z, sc, of), fmaf((float)s.w, sc, of));
            } else {
                const uchar4 s = __ldg(reinterpret_cast<const uchar4*>(reinterpret_cast<const uint8_t*>(base) + off));
                v = make_float4((float)s.x * sc, (float)s.y * sc, (float)s.z * sc, (float)s.w * sc);
            }
            *reinterpret_cast<float4*>(&sG[r][4 * c4]) = v;
        }
    } else {
        for (int i = threadIdx.x; i < GH * GW; i += 256) {
            const int r = i / GW, c = i - r * GW;
            const int gy = reflect101(y0 - 4 + r, hf), gx = reflect101(x0 - 4 + c, wf);
            sG[r][c] = load_scalar<KIND>(base, (size_t)gy * row_stride + gx, sc, of);
        }
    }
}

struct LevelKArgs {
    const void* g;            // input planes (f32 / int16 / u8)
    size_t in_plane;          // elements between planes
    int in_row;               // elements between rows
    float sc[3], of[3];       // per-channel affine for int16 / u8 inputs
    int channels;
    Level lf, lc;
    float* g_next;
    float* hi; float* lo; float* m;
    int first, band;
    double c_hi, omc_hi, c_lo, omc_lo;
    float gain;
    int in_vec_ok;            // u8 rows are 4-byte aligned
};

// PREFETCH (with USE_TMA): the tile's two state planes are requested as bulk-tensor copies at kernel entry, together
// with the input window, and only waited for in the last phase — the fused kernel is latency-bound (B200 probe:
// removing 16 % of its bytes did not shorten it), so what matters is how many bytes each CTA keeps in flight.
template <int KIND, bool USE_TMA, bool PREFETCH>
__global__ void __launch_bounds__(256) k_level(const LevelKArgs a, const __grid_constant__ CUtensorMap tmap,
                                               const __grid_constant__ CUtensorMap tmap_hi,
                                               const __grid_constant__ CUtensorMap tmap_lo) {
    __shared__ __align__(128) float sG[GH][GW];
    __shared__ __align__(16) float sH[GH][DP];
    __shared__ __align__(16) float sD[DH][DP];
    __shared__ __align__(128) float sS[PREFETCH ? 2 : 1][PREFETCH ? TH : 1][PREFETCH ? TW : 4];   // hi / lo tiles
    __shared__ __align__(8) uint64_t tma_bar;
    __shared__ __align__(8) uint64_t st_bar;
    const bool prefetch = PREFETCH && a.band && !a.first;
    const int plane = blockIdx.z;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const int wf = a.lf.w, hf = a.lf.h, wc = a.lc.w, hc = a.lc.h;
    const bool interior = x0 >= 4 && x0 + TW + 4 <= wf && y0 >= 4 && y0 + TH + 3 <= hf && (KIND != IN_U8 || a.in_vec_ok);
    const int ch = plane % a.channels;
    const void* base;
    if (KIND == IN_F32) base = reinterpret_cast<const float*>(a.g) + (size_t)plane * a.in_plane;
    else if (KIND == IN_LAB16) base = reinterpret_cast<const short*>(a.g) + (size_t)plane * a.in_plane;
    else base = reinterpret_cast<const uint8_t*>(a.g) + (size_t)plane * a.in_plane;
    if (USE_TMA) {
        // The (GH x GW) window of this plane is fetched by ONE bulk-tensor copy issued by one thread; the
        // TMA unit zero-fills whatever lies outside the level, and border tiles then patch those cells with
        // BORDER_REFLECT_101 copies taken from inside the window.
        if (threadIdx.x == 0) {
            mbar_init(&tma_bar, 1);
            if (PREFETCH) mbar_init(&st_bar, 1);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            mbar_expect_tx(&tma_bar, GH * GW * sizeof(float));
            tma_load_3d(&sG[0][0], &tmap, x0 - 4, y0 - 4, plane, &tma_bar);
            if (prefetch) {
                mbar_expect_tx(&st_bar, 2 * TH * TW * sizeof(float));
                tma_load_3d(&sS[0][0][0], &tmap_hi, x0, y0, plane, &st_bar);
                tma_load_3d(&sS[PREFETCH ? 1 : 0][0][0], &tmap_lo, x0, y0, plane, &st_bar);
            }
        }
        mbar_wait(&tma_bar, 0);
        if (!interior) {
            __syncthreads();
            float fix[(GH * GW + 255) / 256];
            int n = 0;
            for (int i = threadIdx.x; i < GH * GW; i += 256, ++n) {
                const int r = i / GW, c = i - r * GW;
                const int gy = y0 - 4 + r, gx = x0 - 4 + c;
                int rr = reflect101(gy, hf) - (y0 - 4), cc = reflect101(gx, wf) - (x0 - 4);
                rr = rr < 0 ? 0 : (rr > GH - 1 ? GH - 1 : rr);
                cc = cc < 0 ? 0 : (cc > GW - 1 ? GW - 1 : cc);
                fix[n] = sG[rr][cc];
            }
            __syncthreads();
            n = 0;
            for (int i = threadIdx.x; i < GH * GW; i += 256, ++n) {
                const int r = i / GW, c = i - r * GW;
                sG[r][c] = fix[n];
            }
        }
    } else {
        const float scv = ch == 0 ? a.sc[0] : (ch == 1 ? a.sc[1] : a.sc[2]);
        const float ofv = ch == 0 ? a.of[0] : (ch == 1 ? a.of[1] : a.of[2]);
        load_fine_window<KIND>(sG, base, a.in_row, wf, hf, x0, y0, interior, scv, ofv);
    }
    __syncthreads();

    // pyrDown row pass: sH[r][j] for the coarse columns of the window (pairs of columns per item)
    if (interior) {
        for (int i = threadIdx.x; i < GH * (DW / 2); i += 256) {
            const int r = i / (DW / 2), jp = i - r * (DW / 2);
            const float4 u = *reinterpret_cast<const float4*>(&sG[r][4 * jp]);
            const float4 v = *reinterpret_cast<const float4*>(&sG[r][4 * jp + 4]);
            float2 o;
            o.x = down5(u.x, u.y, u.z, u.w, v.x);
            o.y = down5(u.z, u.w, v.x, v.y, v.z);
            *reinterpret_cast<float2*>(&sH[r][2 * jp]) = o;
        }
    } else {
        for (int i = threadIdx.x; i < GH * DW; i += 256) {
            const int r = i / DW, j = i - r * DW;
            const int im = upsrc(x0 / 2 - 1 + j, wc);
            int c = 2 * im - x0 + 4;
            c = c < 2 ? 2 : (c > GW - 4 ? GW - 4 : c);
            sH[r][j] = down5(sG[r][c - 2], sG[r][c - 1], sG[r][c], sG[r][c + 1], sG[r][c + 2]);
        }
    }
    __syncthreads();
    // pyrDown column pass -> coarse window D (pyrUp's border rule pre-applied); store G_{l+1}
    float* __restrict__ gn = a.g_next + (size_t)plane * a.lc.plane;
    if (interior) {
        for (int i = threadIdx.x; i < (DH / 2) * DW; i += 256) {
            const int kp = i / DW, j = i - kp * DW;
            const int r = 4 * kp;  // rows r..r+6 feed coarse rows 2kp, 2kp+1
            const float f0 = sH[r][j], f1 = sH[r + 1][j], f2 = sH[r + 2][j], f3 = sH[r + 3][j], f4 = sH[r + 4][j],
                        f5 = sH[r + 5][j], f6 = sH[r + 6][j];
            const float d0 = down5(f0, f1, f2, f3, f4) * kInv256, d1 = down5(f2, f3, f4, f5, f6) * kInv256;
            sD[2 * kp][j] = d0;
            sD[2 * kp + 1][j] = d1;
            if (j >= 1 && j <= TW / 2) {
                const int ix = x0 / 2 - 1 + j;
                const int iy = y0 / 2 - 1 + 2 * kp;
                if (kp >= 1) gn[(size_t)iy * a.lc.pitch + ix] = d0;             // k = 2kp in [1,16] <=> kp >= 1
                if (kp <= DH / 2 - 2) gn[(size_t)(iy + 1) * a.lc.pitch + ix] = d1;  // k = 2kp+1 <= 16
            }
        }
    } else {
        for (int i = threadIdx.x; i < DH * DW; i += 256) {
            const int k = i / DW, j = i - k * DW;
            const int iy = y0 / 2 - 1 + k, ix = x0 / 2 - 1 + j;
            const int imy = upsrc(iy, hc);
            int r = 2 * imy - y0 + 4;
            r = r < 2 ? 2 : (r > GH - 3 ? GH - 3 : r);
            const float v = down5(sH[r - 2][j], sH[r - 1][j], sH[r][j], sH[r + 1][j], sH[r + 2][j]) * kInv256;
            sD[k][j] = v;
            if (k >= 1 && k <= TH / 2 && j >= 1 && j <= TW / 2 && iy < hc && ix < wc) gn[(size_t)iy * a.lc.pitch + ix] = v;
        }
    }
    if (!a.band) return;
    __syncthreads();

    // pyrUp + band + temporal filter: thread (tx, ty) owns fine pixels x = 4tx..4tx+3, y = 2ty, 2ty+1
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float up[2][4];
    {
        float e[3][4];  // pyrUp row pass for coarse rows ty, ty+1, ty+2 (window rows), fine cols 4tx..4tx+3
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const float2 p0 = *reinterpret_cast<const float2*>(&sD[ty + q][2 * tx]);
            const float2 p1 = *reinterpret_cast<const float2*>(&sD[ty + q][2 * tx + 2]);
            e[q][0] = p0.x + p0.y * 6.0f + p1.x;
            e[q][1] = (p0.y + p1.x) * 4.0f;
            e[q][2] = p0.y + p1.x * 6.0f + p1.y;
            e[q][3] = (p1.x + p1.y) * 4.0f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            up[0][i] = (e[0][i] + e[1][i] * 6.0f + e[2][i]) * kInv64;
            up[1][i] = ((e[1][i] + e[2][i]) * 4.0f) * kInv64;
        }
    }
    float* __restrict__ hi = a.hi + (size_t)plane * a.lf.plane;
    float* __restrict__ lo = a.lo + (size_t)plane * a.lf.plane;
    float* __restrict__ m = a.m ? a.m + (size_t)plane * a.lf.plane : nullptr;
    const int gx = x0 + 4 * tx;
    if (prefetch) mbar_wait(&st_bar, 0);   // every thread observes the copy's completion itself before reading sS
#pragma unroll
    for (int ry = 0; ry < 2; ++ry) {
        const int gy = y0 + 2 * ty + ry;
        if (gy >= hf || gx >= wf) continue;
        const float4 gv = *reinterpret_cast<const float4*>(&sG[2 * ty + ry + 4][4 * tx + 4]);
        float band[4] = {gv.x - up[ry][0], gv.y - up[ry][1], gv.z - up[ry][2], gv.w - up[ry][3]};
        const size_t o = (size_t)gy * a.lf.pitch + gx;
        // rows are padded to a multiple of 32 floats, so a full float4 at gx < wf is always in-bounds
        if (a.first) {
            const float4 b4 = make_float4(band[0], band[1], band[2], band[3]);
            *reinterpret_cast<float4*>(hi + o) = b4;
            *reinterpret_cast<float4*>(lo + o) = b4;
        } else {
            float4 h4, l4;
            if (prefetch) {
                h4 = *reinterpret_cast<const float4*>(&sS[0][PREFETCH ? 2 * ty + ry : 0][PREFETCH ? 4 * tx : 0]);
                l4 = *reinterpret_cast<const float4*>(&sS[PREFETCH ? 1 : 0][PREFETCH ? 2 * ty + ry : 0][PREFETCH ? 4 * tx : 0]);
            } else {
                h4 = *reinterpret_cast<const float4*>(hi + o);
                l4 = *reinterpret_cast<const float4*>(lo + o);
            }
            float nh[4] = {h4.x, h4.y, h4.z, h4.w}, nl[4] = {l4.x, l4.y, l4.z, l4.w}, mm[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                nh[i] = ema(nh[i], band[i], a.omc_hi, a.c_hi);
                nl[i] = ema(nl[i], band[i], a.omc_lo, a.c_lo);
                mm[i] = (nh[i] - nl[i]) * a.gain;
            }
            *reinterpret_cast<float4*>(hi + o) = make_float4(nh[0], nh[1], nh[2], nh[3]);
            *reinterpret_cast<float4*>(lo + o) = make_float4(nl[0], nl[1], nl[2], nl[3]);
            if (m) *reinterpret_cast<float4*>(m + o) = make_float4(mm[0], mm[1], mm[2], mm[3]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// down_strip: pure cv::pyrDown (level 0 of the production path, Gaussian chain of Color) with the row
// pass in registers + warp shuffles and the column pass as a register sliding window — no shared
// memory, no per-pixel index arithmetic.  One warp = a strip of 128 fine columns (lane = 4 fine
// columns = 2 coarse columns); lanes 0 and 31 only provide the halo, so strips advance by 120 columns
// and no lane ever needs a divergent extra load.  Each warp walks DS_ROWS coarse rows top to bottom,
// loading four fine rows ahead of their use.
// ------------------------------------------------------------------------------------------------
constexpr int DS_ROWS = 16;   // coarse rows per warp
constexpr int DS_WARPS = 4;   // warps per CTA (consecutive row chunks of the same strip)
constexpr int DS_COLS = 120;  // fine columns produced per strip (lanes 1..30)

struct DsRaw { float v0, v1, v2, v3; };   // one fine row as seen by one lane (before the row pass)
struct DsRow { float h0, h1; };

template <int KIND>
__device__ __forceinline__ DsRaw ds_load(const void* base, size_t row_off, int gx, int wf, bool fast, float sc, float of) {
    DsRaw r;
    if (fast) {
        if (KIND == IN_F32) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + row_off + gx));
            r.v0 = t.x; r.v1 = t.y; r.v2 = t.z; r.v3 = t.w;
        } else if (KIND == IN_LAB16) {
            const short4 t = __ldg(reinterpret_cast<const short4*>(reinterpret_cast<const short*>(base) + row_off + gx));
            r.v0 = fmaf((float)t.x, sc, of); r.v1 = fmaf((float)t.y, sc, of); r.v2 = fmaf((float)t.z, sc, of); r.v3 = fmaf((float)t.w, sc, of);
        } else {
            const uchar4 t = __ldg(reinterpret_cast<const uchar4*>(reinterpret_cast<const uint8_t*>(base) + row_off + gx));
            r.v0 = (float)t.x * sc; r.v1 = (float)t.y * sc; r.v2 = (float)t.z * sc; r.v3 = (float)t.w * sc;
        }
    } else {   // columns outside [0, wf): BORDER_REFLECT_101
        r.v0 = load_scalar<KIND>(base, row_off + reflect101(gx, wf), sc, of);
        r.v1 = load_scalar<KIND>(base, row_off + reflect101(gx + 1, wf), sc, of);
        r.v2 = load_scalar<KIND>(base, row_off + reflect101(gx + 2, wf), sc, of);
        r.v3 = load_scalar<KIND>(base, row_off + reflect101(gx + 3, wf), sc, of);
    }
    return r;
}

// Row pass of cv::pyrDown: the two left / one right neighbour values come from the adjacent lanes.
__device__ __forceinline__ DsRow ds_rowpass(const DsRaw& r) {
    const float a0 = __shfl_up_sync(0xffffffffu, r.v2, 1), a1 = __shfl_up_sync(0xffffffffu, r.v3, 1);
    const float b0 = __shfl_down_sync(0xffffffffu, r.v0, 1);
    DsRow o;
    o.h0 = down5(a0, a1, r.v0, r.v1, r.v2);
    o.h1 = down5(r.v0, r.v1, r.v2, r.v3, b0);
    return o;
}

struct DownArgs {
    const void* g; size_t in_plane; int in_row; int channels;
    float sc[3], of[3];
    Level lf, lc;
    float* g_next;
    int in_vec_ok;
};

template <int KIND>
__global__ void __launch_bounds__(32 * DS_WARPS) k_down_strip(const DownArgs a) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int plane = blockIdx.z;
    const int wf = a.lf.w, hf = a.lf.h, wc = a.lc.w, hc = a.lc.h;
    const int gx = blockIdx.x * DS_COLS - 4 + lane * 4;               // first fine column of this lane (multiple of 4)
    const int k0 = (blockIdx.y * DS_WARPS + warp) * DS_ROWS;          // first coarse row of this warp
    if (k0 >= hc) return;
    const int ch = plane % a.channels;
    const float sc = ch == 0 ? a.sc[0] : (ch == 1 ? a.sc[1] : a.sc[2]);   // no dynamic indexing of the param struct
    const float of = ch == 0 ? a.of[0] : (ch == 1 ? a.of[1] : a.of[2]);
    const void* base;
    if (KIND == IN_F32) base = reinterpret_cast<const float*>(a.g) + (size_t)plane * a.in_plane;
    else if (KIND == IN_LAB16) base = reinterpret_cast<const short*>(a.g) + (size_t)plane * a.in_plane;
    else base = reinterpret_cast<const uint8_t*>(a.g) + (size_t)plane * a.in_plane;
    const bool fast = gx >= 0 && (gx + 4 <= wf) && a.in_vec_ok;       // whole vector inside the row
    float* __restrict__ out = a.g_next + (size_t)plane * a.lc.plane;
    const int jx = gx >> 1;                                           // first coarse column of this lane
    const bool writer = lane >= 1 && lane <= 30 && jx < wc;
    const int k_end = min(k0 + DS_ROWS, hc);

    // p1..p4 / q1..q4 = row-pass results of fine rows 2k-2 .. 2k+1 for the lane's two coarse columns.
    // Four fine rows are loaded per iteration before any of them is consumed (memory-level parallelism),
    // producing two coarse rows.
#define DS_LOAD(row) ds_load<KIND>(base, (size_t)reflect101((row), hf) * a.in_row, gx, wf, fast, sc, of)
    float p1, p2, p3, p4, q1, q2, q3, q4;
    {
        const DsRaw a1 = DS_LOAD(2 * k0 - 2), a2 = DS_LOAD(2 * k0 - 1), a3 = DS_LOAD(2 * k0), a4 = DS_LOAD(2 * k0 + 1);
        const DsRow r1 = ds_rowpass(a1), r2 = ds_rowpass(a2), r3 = ds_rowpass(a3), r4 = ds_rowpass(a4);
        p1 = r1.h0; q1 = r1.h1; p2 = r2.h0; q2 = r2.h1; p3 = r3.h0; q3 = r3.h1; p4 = r4.h0; q4 = r4.h1;
    }
    for (int k = k0; k < k_end; k += 2) {
        const DsRaw ra = DS_LOAD(2 * k + 2), rb = DS_LOAD(2 * k + 3), rc = DS_LOAD(2 * k + 4), rd = DS_LOAD(2 * k + 5);
        const DsRow ha = ds_rowpass(ra), hb = ds_rowpass(rb), hc_ = ds_rowpass(rc), hd = ds_rowpass(rd);
        if (writer) {
            const float d0 = down5(p1, p2, p3, p4, ha.h0) * kInv256, d1 = down5(q1, q2, q3, q4, ha.h1) * kInv256;
            float* q = out + (size_t)k * a.lc.pitch + jx;
            if (jx + 1 < wc) *reinterpret_cast<float2*>(q) = make_float2(d0, d1);
            else q[0] = d0;
            if (k + 1 < k_end) {
                const float e0 = down5(p3, p4, ha.h0, hb.h0, hc_.h0) * kInv256, e1 = down5(q3, q4, ha.h1, hb.h1, hc_.h1) * kInv256;
                q += a.lc.pitch;
                if (jx + 1 < wc) *reinterpret_cast<float2*>(q) = make_float2(e0, e1);
                else q[0] = e0;
            }
        }
        p1 = ha.h0; p2 = hb.h0; p3 = hc_.h0; p4 = hd.h0;
        q1 = ha.h1; q2 = hb.h1; q3 = hc_.h1; q4 = hd.h1;
    }
#undef DS_LOAD
}

// ------------------------------------------------------------------------------------------------
// ingest_lab: u8 BGR -> Lab (exact OpenCV LUT) -> { Lab16 planes for egress, G1 = pyrDown(Lab) } in one
// pass.  Same strip structure as down_strip (row pass by shuffles, column pass as a register window),
// with the three Lab channels carried together.  The kernel is bound by the divergent LUT gathers (L1 tag
// lookups) and by issue slots, not by HBM: each pixel costs two 256-bit gathers (LabLutCell) and ~80 instructions;
// the next row's 12 input bytes per lane are requested before the current row is converted.
// ------------------------------------------------------------------------------------------------
constexpr int IG_ROWS = 32;   // coarse rows per warp (halo rows re-convert 4 of 68 fine rows)

struct IngestArgs {
    const uint8_t* in; size_t in_step, in_lane_stride;
    int w, h, aligned;
    const LabLutCell* lut;
    int16_t* lab; int pitch16; size_t plane16;
    float* g1; Level l1;
};

struct IgRaw { uint32_t w0, w1, w2; };   // 4 BGR pixels of one lane

__device__ __forceinline__ IgRaw ig_load(const IngestArgs& a, const uint8_t* frame, int row, int gx, bool fast) {
    const uint8_t* p = frame + (size_t)reflect101(row, a.h) * a.in_step;
    IgRaw r;
    if (fast) {
        const uint32_t* q = reinterpret_cast<const uint32_t*>(p + (size_t)gx * 3);
        r.w0 = __ldg(q); r.w1 = __ldg(q + 1); r.w2 = __ldg(q + 2);
    } else {
        uint32_t px[12];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint8_t* q = p + (size_t)reflect101(gx + i, a.w) * 3;
            px[3 * i] = __ldg(q); px[3 * i + 1] = __ldg(q + 1); px[3 * i + 2] = __ldg(q + 2);
        }
        r.w0 = px[0] | (px[1] << 8) | (px[2] << 16) | (px[3] << 24);
        r.w1 = px[4] | (px[5] << 8) | (px[6] << 16) | (px[7] << 24);
        r.w2 = px[8] | (px[9] << 8) | (px[10] << 16) | (px[11] << 24);
    }
    return r;
}

// converts the lane's 4 pixels of fine row `row`, optionally stores Lab16, returns the row pass of the three channels
__device__ __forceinline__ void ig_row(const IngestArgs& a, const IgRaw raw, int row, int gx, bool own, int16_t* lab_lane,
                                       float (&hL)[2], float (&hA)[2], float (&hB)[2]) {
    uint32_t px[12];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        px[i] = (raw.w0 >> (8 * i)) & 0xff;
        px[4 + i] = (raw.w1 >> (8 * i)) & 0xff;
        px[8 + i] = (raw.w2 >> (8 * i)) & 0xff;
    }
    int sL[4], sA[4], sB[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
        lab_fixed_from_q(lab_q_of_u8((int)px[3 * i]), lab_q_of_u8((int)px[3 * i + 1]), lab_q_of_u8((int)px[3 * i + 2]), a.lut, sL[i], sA[i], sB[i]);
    if (own) {   // this warp owns the row and the lane owns the columns: emit the Lab16 planes
        int16_t* o = lab_lane + (size_t)row * a.pitch16 + gx;
        *reinterpret_cast<short4*>(o) = make_short4((short)sL[0], (short)sL[1], (short)sL[2], (short)sL[3]);
        *reinterpret_cast<short4*>(o + a.plane16) = make_short4((short)sA[0], (short)sA[1], (short)sA[2], (short)sA[3]);
        *reinterpret_cast<short4*>(o + 2 * a.plane16) = make_short4((short)sB[0], (short)sB[1], (short)sB[2], (short)sB[3]);
    }
    DsRaw r;
    DsRow o;
    r.v0 = (float)sL[0] * (100.0f / 16384.0f); r.v1 = (float)sL[1] * (100.0f / 16384.0f);
    r.v2 = (float)sL[2] * (100.0f / 16384.0f); r.v3 = (float)sL[3] * (100.0f / 16384.0f);
    o = ds_rowpass(r); hL[0] = o.h0; hL[1] = o.h1;
    r.v0 = fmaf((float)sA[0], 1.0f / 64.0f, -128.0f); r.v1 = fmaf((float)sA[1], 1.0f / 64.0f, -128.0f);
    r.v2 = fmaf((float)sA[2], 1.0f / 64.0f, -128.0f); r.v3 = fmaf((float)sA[3], 1.0f / 64.0f, -128.0f);
    o = ds_rowpass(r); hA[0] = o.h0; hA[1] = o.h1;
    r.v0 = fmaf((float)sB[0], 1.0f / 64.0f, -128.0f); r.v1 = fmaf((float)sB[1], 1.0f / 64.0f, -128.0f);
    r.v2 = fmaf((float)sB[2], 1.0f / 64.0f, -128.0f); r.v3 = fmaf((float)sB[3], 1.0f / 64.0f, -128.0f);
    o = ds_rowpass(r); hB[0] = o.h0; hB[1] = o.h1;
}

template <int WARPS>
__global__ void __launch_bounds__(32 * WARPS) k_ingest_lab(const IngestArgs a) {
    const int lane_id = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lane = blockIdx.z;                                       // stream
    const int gx = blockIdx.x * DS_COLS - 4 + lane_id * 4;
    const int k0 = (blockIdx.y * WARPS + warp) * IG_ROWS;
    const int wc = a.l1.w, hc = a.l1.h;
    if (k0 >= hc) return;
    const int k_end = min(k0 + IG_ROWS, hc);
    const uint8_t* frame = a.in + (size_t)lane * a.in_lane_stride;
    int16_t* lab_lane = a.lab + (size_t)(lane * 3) * a.plane16;
    const bool fast = gx >= 0 && gx + 4 <= a.w && a.aligned;
    const bool col_owner = lane_id >= 1 && lane_id <= 30 && gx < a.w;
    const int jx = gx >> 1;
    const bool writer = lane_id >= 1 && lane_id <= 30 && jx < wc;
    float* __restrict__ oL = a.g1 + (size_t)(lane * 3) * a.l1.plane;

    // window[c][i] = row pass of fine row (2k-2+i), channel c, for the lane's two coarse columns
    float wL[4][2], wA[4][2], wB[4][2];
    IgRaw nxt = ig_load(a, frame, 2 * k0 - 2, gx, fast);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int row = 2 * k0 - 2 + i;
        const IgRaw cur = nxt;
        nxt = ig_load(a, frame, row + 1, gx, fast);
        ig_row(a, cur, row, gx, col_owner && row >= 2 * k0 && row < a.h, lab_lane, wL[i], wA[i], wB[i]);
    }
    for (int k = k0; k < k_end; ++k) {
        float nL[2], nA[2], nB[2];
        {
            const int row = 2 * k + 2;
            const IgRaw cur = nxt;
            nxt = ig_load(a, frame, row + 1, gx, fast);
            ig_row(a, cur, row, gx, col_owner && row < 2 * k_end && row < a.h, lab_lane, nL, nA, nB);
        }
        if (writer) {
            float* q = oL + (size_t)k * a.l1.pitch + jx;
            const bool two = jx + 1 < wc;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float (*wnd)[2] = c == 0 ? wL : (c == 1 ? wA : wB);
                const float* nn = c == 0 ? nL : (c == 1 ? nA : nB);
                const float d0 = down5(wnd[0][0], wnd[1][0], wnd[2][0], wnd[3][0], nn[0]) * kInv256;
                const float d1 = down5(wnd[0][1], wnd[1][1], wnd[2][1], wnd[3][1], nn[1]) * kInv256;
                float* qc = q + (size_t)c * a.l1.plane;
                if (two) *reinterpret_cast<float2*>(qc) = make_float2(d0, d1);
                else qc[0] = d0;
            }
        }
        // slide by two fine rows: rows 2k .. 2k+3 become the next window
        float mL[2], mA[2], mB[2];
        {
            const int row = 2 * k + 3;
            const bool need = k + 1 < k_end;   // the last iteration's extra row is never used
            if (need) {
                const IgRaw cur = nxt;
                nxt = ig_load(a, frame, row + 1, gx, fast);
                ig_row(a, cur, row, gx, col_owner && row < 2 * k_end && row < a.h, lab_lane, mL, mA, mB);
            } else { mL[0] = mL[1] = mA[0] = mA[1] = mB[0] = mB[1] = 0.f; }
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            wL[0][j] = wL[2][j]; wL[1][j] = wL[3][j]; wL[2][j] = nL[j]; wL[3][j] = mL[j];
            wA[0][j] = wA[2][j]; wA[1][j] = wA[3][j]; wA[2][j] = nA[j]; wA[3][j] = mA[j];
            wB[0][j] = wB[2][j]; wB[1][j] = wB[3][j]; wB[2][j] = nB[j]; wB[3][j] = mB[j];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// collapse: cur_l = pyrUp(cur_{l+1}) + m_l.  The band-passed, amplified band m_l = gain_l * (hi_l - lo_l)
// (TemporalFilter.cpp:21, MagnifyCore.hpp:127-134) is either the plane the level kernel stored (then `out` may be
// that same plane: every thread reads its pixels before it writes them) or, with option band_from_state, rebuilt
// from the two state planes the level kernel has just written (same f32 subtract and multiply).  Tile 64 x 32,
// thread block 4 x 2 (same register pyrUp as the level kernel), 128-bit accesses.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float band_at(const BandSrc& b, size_t off) {
    const float v = __ldg(b.a + off);
    return b.b ? band_of(v, __ldg(b.b + off), b.gain) : v;
}

__global__ void __launch_bounds__(256) k_collapse(Level lf, Level lc, BandSrc fine, BandSrc coarse, float* out, int plane_step) {
    __shared__ __align__(16) float sD[DH][DP];
    const int plane = blockIdx.z * plane_step;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const size_t cbase = (size_t)plane * lc.plane;
    for (int i = threadIdx.x; i < DH * DW; i += 256) {
        const int k = i / DW, j = i - k * DW;
        const int iy = upsrc(y0 / 2 - 1 + k, lc.h), ix = upsrc(x0 / 2 - 1 + j, lc.w);
        sD[k][j] = band_at(coarse, cbase + (size_t)iy * lc.pitch + ix);
    }
    __syncthreads();
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int gx = x0 + 4 * tx;
    if (gx >= lf.w) return;
    float e[3][4];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        const float2 p0 = *reinterpret_cast<const float2*>(&sD[ty + q][2 * tx]);
        const float2 p1 = *reinterpret_cast<const float2*>(&sD[ty + q][2 * tx + 2]);
        e[q][0] = up3(p0.x, p0.y, p1.x);
        e[q][1] = up2(p0.y, p1.x);
        e[q][2] = up3(p0.y, p1.x, p1.y);
        e[q][3] = up2(p1.x, p1.y);
    }
    const size_t fbase = (size_t)plane * lf.plane;
#pragma unroll
    for (int ry = 0; ry < 2; ++ry) {
        const int gy = y0 + 2 * ty + ry;
        if (gy >= lf.h) continue;
        const size_t o = fbase + (size_t)gy * lf.pitch + gx;   // rows padded to 32 floats: a float4 at gx < w is in-bounds
        float4 v = *reinterpret_cast<const float4*>(fine.a + o);   // plain load: `out` may be this very plane
        if (fine.b) {
            const float4 u = __ldg(reinterpret_cast<const float4*>(fine.b + o));
            v.x = band_of(v.x, u.x, fine.gain); v.y = band_of(v.y, u.y, fine.gain); v.z = band_of(v.z, u.z, fine.gain); v.w = band_of(v.w, u.w, fine.gain);
        }
        if (ry == 0) {
            v.x = __fmaf_rn(up3(e[0][0], e[1][0], e[2][0]), kInv64, v.x);   // * 2^-6 is exact: one rounding, in the add
            v.y = __fmaf_rn(up3(e[0][1], e[1][1], e[2][1]), kInv64, v.y);
            v.z = __fmaf_rn(up3(e[0][2], e[1][2], e[2][2]), kInv64, v.z);
            v.w = __fmaf_rn(up3(e[0][3], e[1][3], e[2][3]), kInv64, v.w);
        } else {
            v.x = __fmaf_rn(up2(e[1][0], e[2][0]), kInv64, v.x);
            v.y = __fmaf_rn(up2(e[1][1], e[2][1]), kInv64, v.y);
            v.z = __fmaf_rn(up2(e[1][2], e[2][2]), kInv64, v.z);
            v.w = __fmaf_rn(up2(e[1][3], e[2][3]), kInv64, v.w);
        }
        *reinterpret_cast<float4*>(out + o) = v;
    }
}

// ------------------------------------------------------------------------------------------------
// egress: tile = 64 x 32 output pixels, all channels; thread block of 4 x 2 pixels.
//   cur_1 = pyrUp(cur_2) + m_1 is rebuilt on the tile's level-1 window (34 x 18), then
//   out = convert(input + chroma * pyrUp(cur_1)).
// ------------------------------------------------------------------------------------------------
constexpr int E2W = 20, E2H = 12;   // level-2 window, origin (x0/4-2, y0/4-2)
constexpr int E2P = 20;

struct EgressArgs {
    const uint8_t* in; size_t in_step, in_lane_stride;      // gray input (C == 1)
    const int16_t* lab; int pitch16; size_t plane16;        // Lab16 planes (C == 3)
    uint8_t* out; size_t out_step, out_lane_stride;
    int w0, h0;
    const float4* gtab; LabInvCoeffs coeffs;
    BandSrc m1; Level l1;           // band 1 = gain_1 * (hi_1 - lo_1) rebuilt from the state planes; a == null: no motion
    BandSrc c2; Level l2;           // collapsed level 2 (or band 2 from state when it is the top band); a == null: cur_1 = m_1
    float chroma;
    float* fout;
};

// The pixel stage of egress for the 4 output pixels (gy, gx .. gx+3) of stream `lane`: input (+ motion `up`, the a / b
// planes attenuated by chroma) -> Lab2BGR -> u8 (MagnifyCore.hpp:140-158).  Split into the load of the input samples
// (so that the strip kernel can request them an iteration ahead) and the conversion.
template <int C> struct EgressIn;
template <> struct EgressIn<3> { short4 L, A, B; };
template <> struct EgressIn<1> { uint32_t g; };

template <int C>
__device__ __forceinline__ EgressIn<C> egress_load(const EgressArgs& a, int lane, int gy, int gx);
template <>
__device__ __forceinline__ EgressIn<3> egress_load<3>(const EgressArgs& a, int lane, int gy, int gx) {
    const int16_t* lp = a.lab + (size_t)(lane * 3) * a.plane16 + (size_t)gy * a.pitch16 + gx;
    EgressIn<3> r;
    r.L = __ldg(reinterpret_cast<const short4*>(lp));
    r.A = __ldg(reinterpret_cast<const short4*>(lp + a.plane16));
    r.B = __ldg(reinterpret_cast<const short4*>(lp + 2 * a.plane16));
    return r;
}
template <>
__device__ __forceinline__ EgressIn<1> egress_load<1>(const EgressArgs& a, int lane, int gy, int gx) {
    const uint8_t* p = a.in + (size_t)lane * a.in_lane_stride + (size_t)gy * a.in_step + gx;
    EgressIn<1> r;
    r.g = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (gx + i < a.w0) r.g |= (uint32_t)__ldg(p + i) << (8 * i);
    return r;
}

// `up` holds the pyrUp tap sums BEFORE their 1/64 scale: the scale is exact, so it is folded into the add (L) and
// into the chroma factor (a, b) without changing a bit.  q / f: the row's output pointers at column gx (f may be null).
// MC: channels of the motion image — 3, or 1 (L only) when chroma is 0: the attenuated a and b motion is then +-0 and
// input + motion is the input itself, bit for bit (DESIGN §4), so A and B pass through.
template <int MC>
__device__ __forceinline__ void egress_convert(const EgressArgs& a, uint8_t* q, float* f, int gx, const EgressIn<3>& in, const float (&up)[MC][4]) {
    static_assert(MC == 1 || MC == 3, "motion channels");
    uint8_t o8[12];
    float of[12];
    const short vL[4] = {in.L.x, in.L.y, in.L.z, in.L.w}, vA[4] = {in.A.x, in.A.y, in.A.z, in.A.w}, vB[4] = {in.B.x, in.B.y, in.B.z, in.B.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float L = (float)vL[i] * (100.0f / 16384.0f);
        float A = fmaf((float)vA[i], 1.0f / 64.0f, -128.0f);
        float B = fmaf((float)vB[i], 1.0f / 64.0f, -128.0f);
        if (a.m1.a) {
            // a,b motion planes *= chromAttenuation, then output = input + motion (MagnifyCore.hpp:140-148)
            L = __fmaf_rn(up[0][i], kInv64, L);
            if constexpr (MC == 3) {
                const float chroma64 = a.chroma * kInv64;
                A = __fadd_rn(A, __fmul_rn(up[1][i], chroma64));   // the reference scales the plane, then adds
                B = __fadd_rn(B, __fmul_rn(up[2][i], chroma64));
            }
        }
        float ob, og, orr;
        lab_to_bgr_fast<false, true>(L, A, B, a.coeffs, a.gtab, ob, og, orr);
        of[3 * i] = ob; of[3 * i + 1] = og; of[3 * i + 2] = orr;
        // lab_to_bgr clips to [0,1] before the gamma spline, so the saturating branches of
        // convertTo reduce to a min with 255 (NaN -> 0 by the conversion itself)
        o8[3 * i] = unit01_to_u8(ob); o8[3 * i + 1] = unit01_to_u8(og); o8[3 * i + 2] = unit01_to_u8(orr);
    }
    if (gx + 4 <= a.w0 && ((reinterpret_cast<uintptr_t>(q) & 3) == 0)) {
#pragma unroll
        for (int wd = 0; wd < 3; ++wd)
            reinterpret_cast<uint32_t*>(q)[wd] = (uint32_t)o8[4 * wd] | ((uint32_t)o8[4 * wd + 1] << 8) |
                                                 ((uint32_t)o8[4 * wd + 2] << 16) | ((uint32_t)o8[4 * wd + 3] << 24);
    } else {
#pragma unroll
        for (int i = 0; i < 12; ++i)
            if (gx + i / 3 < a.w0) q[i] = o8[i];
    }
    if (f) {
#pragma unroll
        for (int i = 0; i < 12; ++i)
            if (gx + i / 3 < a.w0) f[i] = of[i];
    }
}
__device__ __forceinline__ void egress_convert(const EgressArgs& a, uint8_t* q, float* f, int gx, const EgressIn<1>& in, const float (&up)[1][4]) {
    uint8_t o8[4];
    float of[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float v = u8_to_unit((uint8_t)((in.g >> (8 * i)) & 0xff));
        if (a.m1.a) v = __fmaf_rn(up[0][i], kInv64, v);
        of[i] = v;
        o8[i] = unit_to_u8(v);
    }
    if (gx + 4 <= a.w0 && ((reinterpret_cast<uintptr_t>(q) & 3) == 0)) {
        *reinterpret_cast<uint32_t*>(q) = (uint32_t)o8[0] | ((uint32_t)o8[1] << 8) | ((uint32_t)o8[2] << 16) | ((uint32_t)o8[3] << 24);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (gx + i < a.w0) q[i] = o8[i];
    }
    if (f) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (gx + i < a.w0) f[i] = of[i];
    }
}

template <int C, int MC>
__device__ __forceinline__ void egress_pixels(const EgressArgs& a, int lane, int gy, int gx, const float (&up)[MC][4]) {
    const EgressIn<C> in = egress_load<C>(a, lane, gy, gx);
    uint8_t* q = a.out + (size_t)lane * a.out_lane_stride + (size_t)gy * a.out_step + (size_t)gx * C;
    float* f = a.fout ? a.fout + (((size_t)lane * a.h0 + gy) * a.w0 + gx) * C : nullptr;
    egress_convert(a, q, f, gx, in, up);
}

// MC: motion channels (1 with C == 3: only the L planes of the band / cur planes are read, see egress_convert).
template <int C, int MC>
__global__ void __launch_bounds__(256) k_egress(const EgressArgs a) {
    __shared__ __align__(16) float sC2[MC][E2H][E2P];
    __shared__ __align__(16) float sT[MC][E2H][DP];    // horizontal pyrUp pass of the level-2 window rows
    __shared__ __align__(16) float sD[MC][DH][DP];
    const int lane = blockIdx.z;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const int w1 = a.l1.w, h1 = a.l1.h;
    if (a.m1.a) {
        // cur_1 = pyrUp(cur_2) + m_1 on the tile's level-1 window; m_1 is the stored band plane, or gain_1 * (hi_1 - lo_1)
        // rebuilt from the two state planes (option band_from_state).  Position (k, j) of the window is
        // level-1 pixel (y1, x1) = (upsrc(y0/2-1+k), upsrc(x0/2-1+j)).  pyrUp is evaluated separably: the
        // horizontal pass of every level-2 window row at the 34 level-1 columns first (sT), then the vertical
        // pass per position — same operation order as evaluating the 3x3 footprint per position, a fraction of
        // the instructions.  Window index of level-2 pixel i is i - (x0/4 - 2); pyrUp's border rule is applied
        // when the level-2 window is loaded (entries hold s[upsrc(i)]).
        const bool has2 = a.c2.a != nullptr;
        const int bx2 = x0 / 4 - 2, by2 = y0 / 4 - 2;
        if (has2) {
            {
                const size_t base2 = (size_t)(lane * C) * a.l2.plane;
                for (int i = threadIdx.x; i < E2H * E2W; i += 256) {
                    const int k = i / E2W, j = i - k * E2W;
                    const int o2 = upsrc(by2 + k, a.l2.h) * a.l2.pitch + upsrc(bx2 + j, a.l2.w);
#pragma unroll
                    for (int ch = 0; ch < MC; ++ch) sC2[ch][k][j] = band_at(a.c2, base2 + (size_t)ch * a.l2.plane + o2);
                }
                __syncthreads();
            }
            for (int i = threadIdx.x; i < E2H * DW; i += 256) {
                const int ky = i / DW, j = i - ky * DW;
                const int x1 = upsrc(x0 / 2 - 1 + j, w1);
                const int jx = (x1 >> 1) - bx2;
                const bool odd = x1 & 1;
                const int r = ky, cm = jx - 1, c0 = jx, cp = jx + 1;   // the window holds s[upsrc(i)]
#pragma unroll
                for (int ch = 0; ch < MC; ++ch) {
                    const float sm = sC2[ch][r][cm], s0 = sC2[ch][r][c0], sp = sC2[ch][r][cp];
                    sT[ch][ky][j] = odd ? up2(s0, sp) : up3(sm, s0, sp);
                }
            }
            __syncthreads();
        }
        const float* __restrict__ ph[MC];
        const float* __restrict__ pl[MC];
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) {
            ph[ch] = a.m1.a + (size_t)(lane * C + ch) * a.l1.plane;
            pl[ch] = a.m1.b ? a.m1.b + (size_t)(lane * C + ch) * a.l1.plane : nullptr;
        }
        const float g1 = a.m1.gain;
        const bool from_state = a.m1.b != nullptr;
        for (int i = threadIdx.x; i < DH * DW; i += 256) {
            const int k = i / DW, j = i - k * DW;
            const int y1 = upsrc(y0 / 2 - 1 + k, h1), x1 = upsrc(x0 / 2 - 1 + j, w1);
            const int o1 = y1 * a.l1.pitch + x1;
            float v[MC];
#pragma unroll
            for (int ch = 0; ch < MC; ++ch) {
                v[ch] = __ldg(ph[ch] + o1);
                if (from_state) v[ch] = band_of(v[ch], __ldg(pl[ch] + o1), g1);
            }
            if (has2) {
                const int ky = (y1 >> 1) - by2;
                const bool odd = y1 & 1;
#pragma unroll
                for (int ch = 0; ch < MC; ++ch) {
                    const float r0 = sT[ch][ky - 1][j], r1 = sT[ch][ky][j], r2 = sT[ch][ky + 1][j];
                    v[ch] = __fmaf_rn(odd ? up2(r1, r2) : up3(r0, r1, r2), kInv64, v[ch]);
                }
            }
#pragma unroll
            for (int ch = 0; ch < MC; ++ch) sD[ch][k][j] = v[ch];
        }
        __syncthreads();
    }
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int gx = x0 + 4 * tx;
    if (gx >= a.w0) return;
    float up[MC][2][4];
    if (a.m1.a) {
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) {
            float e[3][4];
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const float2 p0 = *reinterpret_cast<const float2*>(&sD[ch][ty + q][2 * tx]);
                const float2 p1 = *reinterpret_cast<const float2*>(&sD[ch][ty + q][2 * tx + 2]);
                e[q][0] = up3(p0.x, p0.y, p1.x);
                e[q][1] = up2(p0.y, p1.x);
                e[q][2] = up3(p0.y, p1.x, p1.y);
                e[q][3] = up2(p1.x, p1.y);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                up[ch][0][i] = up3(e[0][i], e[1][i], e[2][i]);   // x 1/64 is applied (exactly) in egress_convert
                up[ch][1][i] = up2(e[1][i], e[2][i]);
            }
        }
    }
#pragma unroll
    for (int ry = 0; ry < 2; ++ry) {
        const int gy = y0 + 2 * ty + ry;
        if (gy >= a.h0) continue;
        float upr[MC][4];
#pragma unroll
        for (int ch = 0; ch < MC; ++ch)
#pragma unroll
            for (int i = 0; i < 4; ++i) upr[ch][i] = up[ch][ry][i];
        egress_pixels<C>(a, lane, gy, gx, upr);
    }
}

// ------------------------------------------------------------------------------------------------
// egress, strip form (default): the same collapse of levels 2 -> 1 -> 0 and pixel stage as k_egress, without shared
// memory, barriers or per-position index arithmetic.  One warp owns a strip of 128 output columns (lane = 4 columns =
// 2 level-1 columns = 1 level-2 column; lanes 0 and 31 only provide the halo, strips advance by 120 columns) and walks
// EG_ROWS output rows top to bottom: horizontal pyrUp passes take their neighbours from the adjacent lanes by shuffle,
// vertical passes are register sliding windows — three horizontally expanded level-2 rows (H2) and three horizontally
// expanded cur_1 rows (E).  Every value is computed by the same operations in the same order as in k_egress (and as
// cv::pyrUp: row pass first), so the two kernels agree bit for bit; pyrUp's border rule (s[-1] := s[1],
// s[n] := s[n-1]) is applied to the shuffled / streamed neighbours.  The kernel is issue-bound (Lab2BGR), not HBM-bound.
// ------------------------------------------------------------------------------------------------
// input samples of one row from running pointers (strip kernel): the three Lab16 plane rows at byte/element offset `off`,
// or four gray bytes of a row
template <int C>
__device__ __forceinline__ EgressIn<C> egress_rows3(const int16_t* const (&p)[C], size_t off);
template <>
__device__ __forceinline__ EgressIn<3> egress_rows3<3>(const int16_t* const (&p)[3], size_t off) {
    EgressIn<3> r;
    r.L = __ldg(reinterpret_cast<const short4*>(p[0] + off));
    r.A = __ldg(reinterpret_cast<const short4*>(p[1] + off));
    r.B = __ldg(reinterpret_cast<const short4*>(p[2] + off));
    return r;
}
template <>
__device__ __forceinline__ EgressIn<1> egress_rows3<1>(const int16_t* const (&)[1], size_t) { return EgressIn<1>{0}; }
template <int C>
__device__ __forceinline__ EgressIn<C> egress_row1(const uint8_t* row, int gx, int w0);
template <>
__device__ __forceinline__ EgressIn<1> egress_row1<1>(const uint8_t* row, int gx, int w0) {
    EgressIn<1> r;
    r.g = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (gx >= 0 && gx + i < w0) r.g |= (uint32_t)__ldg(row + gx + i) << (8 * i);
    return r;
}
template <>
__device__ __forceinline__ EgressIn<3> egress_row1<3>(const uint8_t*, int, int) { return EgressIn<3>{}; }

constexpr int EG_ROWS = 64;   // output rows per warp (a multiple of 4)

template <int C> struct StripM1 { float2 h[C], l[C]; };   // band-1 source of one cur_1 row at the lane's two columns
template <int C> struct StripH2 { float v[C], vb[C], vr[C], vrb[C]; };   // one level-2 row at the lane's column (+ lane 31's right neighbour); b: lo state

// MC: motion channels (1 with C == 3 when chroma is 0): the band / cur loads, both sliding windows and every pyrUp pass
// run on the L planes only, and egress_convert passes A and B through.
template <int C, int MC, int MINB>
__global__ void __launch_bounds__(32, MINB) k_egress_strip(const EgressArgs a) {
    const unsigned full = 0xffffffffu;
    const int lane_id = threadIdx.x;
    const int lane = blockIdx.z;
    const int gx = blockIdx.x * DS_COLS - 4 + lane_id * 4;          // first output column of this lane (multiple of 4)
    const int f0 = blockIdx.y * EG_ROWS;
    if (f0 >= a.h0) return;
    const int f_end = min(f0 + EG_ROWS, a.h0);
    const bool px_owner = lane_id >= 1 && lane_id <= 30 && gx < a.w0;
    if (!a.m1.a) {   // no motion (first frame, or fewer than two levels): conversion only
        float zero[MC][4];
#pragma unroll
        for (int ch = 0; ch < MC; ++ch)
#pragma unroll
            for (int i = 0; i < 4; ++i) zero[ch][i] = 0.0f;
        if (px_owner)
            for (int gy = f0; gy < f_end; ++gy) egress_pixels<C>(a, lane, gy, gx, zero);
        return;
    }
    const int w1 = a.l1.w, h1 = a.l1.h, w2 = a.l2.w, h2 = a.l2.h;
    const int x1a = gx >> 1, x2 = gx >> 2;                           // lane 0 of strip 0: -2, -1
    const bool has2 = a.c2.a != nullptr, from_state = a.m1.b != nullptr, st2 = a.c2.b != nullptr;
    const float g1 = a.m1.gain, g2 = a.c2.gain;
    // clamped columns for the loads of lanes outside the level (their values are never used)
    const int x1l = x1a < 0 ? 0 : (x1a >= w1 ? ((w1 - 1) & ~1) : x1a);
    const int x2l = x2 < 0 ? 0 : (x2 >= w2 ? w2 - 1 : x2);
    const int x2r = x2l + 1 >= w2 ? w2 - 1 : x2l + 1;                // lane 31's right neighbour column
    const int gxl = px_owner ? gx : 0;                               // input column for the (unused) loads of non-owners
    size_t base1[MC], base2[MC];
#pragma unroll
    for (int ch = 0; ch < MC; ++ch) {
        base1[ch] = (size_t)(lane * C + ch) * a.l1.plane + x1l;
        base2[ch] = (size_t)(lane * C + ch) * a.l2.plane;
    }

    // ---- loads; the lines of the next iteration are requested into L1 while the current one is computed ----
    auto row1 = [&](int y1) { return (size_t)(y1 < h1 ? y1 : h1 - 1) * a.l1.pitch; };   // rows past the end are border copies
    auto ld_m1 = [&](int y1) {
        StripM1<MC> m;
        const size_t ro = row1(y1);
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) {
            m.h[ch] = __ldg(reinterpret_cast<const float2*>(a.m1.a + base1[ch] + ro));
            m.l[ch] = from_state ? __ldg(reinterpret_cast<const float2*>(a.m1.b + base1[ch] + ro)) : make_float2(0.f, 0.f);
        }
        return m;
    };
    auto pf_m1 = [&](int y1) {
        const size_t ro = row1(y1);
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) {
            prefetch_l1(a.m1.a + base1[ch] + ro);
            if (from_state) prefetch_l1(a.m1.b + base1[ch] + ro);
        }
    };
    auto ld_h2 = [&](int y2) {
        StripH2<MC> r;
        const size_t ro = (size_t)upsrc(y2, h2) * a.l2.pitch;
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) {
            r.v[ch] = r.vb[ch] = r.vr[ch] = r.vrb[ch] = 0.f;
            if (has2) {
                r.v[ch] = __ldg(a.c2.a + base2[ch] + ro + x2l);
                if (st2) r.vb[ch] = __ldg(a.c2.b + base2[ch] + ro + x2l);
                if (lane_id == 31) {
                    r.vr[ch] = __ldg(a.c2.a + base2[ch] + ro + x2r);
                    if (st2) r.vrb[ch] = __ldg(a.c2.b + base2[ch] + ro + x2r);
                }
            }
        }
        return r;
    };
    auto pf_h2 = [&](int y2) {
        const size_t ro = (size_t)upsrc(y2, h2) * a.l2.pitch;
        if (has2) {
#pragma unroll
            for (int ch = 0; ch < MC; ++ch) {
                prefetch_l1(a.c2.a + base2[ch] + ro + x2l);
                if (st2) prefetch_l1(a.c2.b + base2[ch] + ro + x2l);
            }
        }
    };
    auto pf_in = [&](int gy) {
        if (C == 3) {
            const int16_t* lp = a.lab + (size_t)(lane * 3) * a.plane16 + (size_t)gy * a.pitch16 + gxl;
            prefetch_l1(lp); prefetch_l1(lp + a.plane16); prefetch_l1(lp + 2 * a.plane16);
        } else {
            prefetch_l1(a.in + (size_t)lane * a.in_lane_stride + (size_t)gy * a.in_step + gxl);
        }
    };
    // ---- compute ----
    // The two sliding windows live in shared memory as per-lane rings of three rows (each lane only ever reads back what
    // it stored itself, so no synchronisation is involved): they would otherwise hold 54 registers across the whole
    // pixel stage and halve the number of resident warps of an issue-bound kernel.
    //   sH[i % 3]: horizontally expanded level-2 row i at the lane's two level-1 columns (even, odd)
    //   sE[j % 3]: horizontally expanded cur_1 row j at the lane's four output columns
    __shared__ float2 sH[3][MC][32];
    __shared__ float4 sE[3][MC][32];
    auto slot = [](int r) { return (r + 3) % 3; };      // rows >= -1
    auto expand_h2 = [&](const StripH2<MC>& in, int i) {
        const int sl = slot(i);
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) {
            const float v = st2 ? band_of(in.v[ch], in.vb[ch], g2) : in.v[ch];
            float l = __shfl_up_sync(full, v, 1), r = __shfl_down_sync(full, v, 1);
            if (lane_id == 31) r = st2 ? band_of(in.vr[ch], in.vrb[ch], g2) : in.vr[ch];
            if (x2 == 0) l = r;                    // s[-1] := s[1]
            if (x2 + 1 >= w2) r = v;               // s[w2] := s[w2-1]
            sH[sl][ch][lane_id] = make_float2(up3(l, v, r), up2(v, r));
        }
    };
    // cur_1 row y1 at the lane's two columns = pyrUp(cur_2) + m_1, then its horizontal expansion at the lane's four
    // output columns.  An even row 2i takes level-2 rows (i-1, i, i+1), an odd row 2i+1 rows (i, i+1).
    auto cur1_row = [&](const StripM1<MC>& m, int y1, float (&E)[MC][4]) {
        const bool odd = y1 & 1;
        const int i = y1 >> 1;
        const int sp = slot(odd ? i : i - 1), sq = slot(odd ? i + 1 : i), sr = slot(i + 1);
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) {
            float ca = m.h[ch].x, cb = m.h[ch].y;
            if (from_state) {
                ca = band_of(ca, m.l[ch].x, g1);
                cb = band_of(cb, m.l[ch].y, g1);
            }
            if (has2) {
                const float2 p = sH[sp][ch][lane_id], q = sH[sq][ch][lane_id], r = sH[sr][ch][lane_id];
                ca = __fmaf_rn(odd ? up2(p.x, q.x) : up3(p.x, q.x, r.x), kInv64, ca);
                cb = __fmaf_rn(odd ? up2(p.y, q.y) : up3(p.y, q.y, r.y), kInv64, cb);
            }
            if (x1a + 1 >= w1) cb = ca;                                  // cur_1[w1] := cur_1[w1-1]
            float left = __shfl_up_sync(full, cb, 1), right = __shfl_down_sync(full, ca, 1);
            if (x1a == 0) left = cb;                                     // cur_1[-1] := cur_1[1]
            if (x1a + 2 >= w1) right = cb;
            E[ch][0] = up3(left, ca, cb);
            E[ch][1] = up2(ca, cb);
            E[ch][2] = up3(ca, cb, right);
            E[ch][3] = up2(cb, right);
        }
    };
    auto put_E = [&](int j, const float (&E)[MC][4]) {
        const int sl = slot(j);
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) sE[sl][ch][lane_id] = make_float4(E[ch][0], E[ch][1], E[ch][2], E[ch][3]);
    };

    const int j0 = f0 >> 1;                       // first level-1 row of the chunk (even)
    {
        const int ic = j0 >> 1;
        const StripH2<MC> ra = ld_h2(ic - 1), rb = ld_h2(ic), rc = ld_h2(ic + 1);
        const StripM1<MC> mp = ld_m1(j0 > 0 ? j0 - 1 : 1), m0 = ld_m1(j0);
        pf_m1(j0 + 1);
        pf_in(2 * j0);
        pf_in(min(2 * j0 + 1, a.h0 - 1));
        expand_h2(ra, ic - 1);
        expand_h2(rb, ic);
        expand_h2(rc, ic + 1);
        float E[MC][4];
        // row j0-1 (odd, level-2 rows ic-1, ic); at the top of the image the slot of row -1 is filled with row 1 below
        if (j0 > 0) { cur1_row(mp, j0 - 1, E); put_E(j0 - 1, E); }
        cur1_row(m0, j0, E);
        put_E(j0, E);
    }
    const int j_end = (f_end + 1) >> 1;
    // Running row pointers (advanced once per iteration instead of rebuilt per access): band-1 source rows at the lane's
    // level-1 columns, the input rows at the lane's output columns, the output row.
    const size_t st1 = (size_t)a.l1.pitch, st16 = (size_t)a.pitch16;
    const float* ph[MC];
    const float* pl[MC];
    const int16_t* pin[C];
#pragma unroll
    for (int ch = 0; ch < C; ++ch) {
        if (ch < MC) {
            const size_t ro = row1(j0 + 1);
            ph[ch] = a.m1.a + base1[ch] + ro;
            pl[ch] = from_state ? a.m1.b + base1[ch] + ro : ph[ch];
        }
        pin[ch] = C == 3 ? a.lab + (size_t)(lane * 3 + ch) * a.plane16 + (size_t)(2 * j0) * st16 + gxl : nullptr;
    }
    const uint8_t* pg = C == 1 ? a.in + (size_t)lane * a.in_lane_stride + (size_t)(2 * j0) * a.in_step : nullptr;   // gray input row
    uint8_t* pq = a.out + (size_t)lane * a.out_lane_stride + (size_t)(2 * j0) * a.out_step + (size_t)gx * C;
    int sm = slot(j0 - 1), s0 = slot(j0), sp = slot(j0 + 1);           // ring slots of cur_1 rows j-1, j, j+1
    for (int j = j0; j < j_end; ++j) {
        const int jn = j + 1;
        const bool two = 2 * j + 1 < f_end;                            // the chunk may end on an even row
        // what this iteration consumes (requested into L1 by the previous one) ...
        StripM1<MC> cm;
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) {
            cm.h[ch] = __ldg(reinterpret_cast<const float2*>(ph[ch]));
            cm.l[ch] = from_state ? __ldg(reinterpret_cast<const float2*>(pl[ch])) : make_float2(0.f, 0.f);
        }
        StripH2<MC> chh;
        if (!(jn & 1) && jn < h1) chh = ld_h2((jn >> 1) + 1);
        EgressIn<C> in0, in1;
        if (C == 3) {
            in0 = egress_rows3<C>(pin, 0);
            in1 = egress_rows3<C>(pin, two ? st16 : 0);
        } else {
            in0 = egress_row1<C>(pg, gx, a.w0);
            in1 = egress_row1<C>(two ? pg + a.in_step : pg, gx, a.w0);
        }
        // ... and the requests for the next one: cur_1 row j+2, the level-2 row that enters the window with it, the inputs
        if (jn < j_end) {
            const bool adv1 = jn + 1 < h1;
            if (jn & 1) pf_h2(((jn + 1) >> 1) + 1);
#pragma unroll
            for (int ch = 0; ch < C; ++ch) {
                if (ch < MC) {
                    if (adv1) { ph[ch] += st1; pl[ch] += st1; }
                    prefetch_l1(ph[ch]);
                    if (from_state) prefetch_l1(pl[ch]);
                }
                if (C == 3) {
                    pin[ch] += 2 * st16;
                    prefetch_l1(pin[ch]);
                    if (2 * jn + 1 < a.h0) prefetch_l1(pin[ch] + st16);
                }
            }
            if (C == 1) { pg += 2 * a.in_step; prefetch_l1(pg + gxl); }
        }
        // row j+1 of cur_1 (or its border copy) -> Ep
        float Ep[MC][4];
        if (jn >= h1) {
#pragma unroll
            for (int ch = 0; ch < MC; ++ch) {
                const float4 e = sE[s0][ch][lane_id];
                Ep[ch][0] = e.x; Ep[ch][1] = e.y; Ep[ch][2] = e.z; Ep[ch][3] = e.w;
            }
        } else {
            if (!(jn & 1)) expand_h2(chh, (jn >> 1) + 1);     // an even row moves the level-2 window to centre jn / 2
            cur1_row(cm, jn, Ep);
        }
#pragma unroll
        for (int ch = 0; ch < MC; ++ch) sE[sp][ch][lane_id] = make_float4(Ep[ch][0], Ep[ch][1], Ep[ch][2], Ep[ch][3]);
        if (j == 0) {                                         // cur_1[-1] := cur_1[1]
#pragma unroll
            for (int ch = 0; ch < MC; ++ch) sE[sm][ch][lane_id] = make_float4(Ep[ch][0], Ep[ch][1], Ep[ch][2], Ep[ch][3]);
        }
        if (px_owner) {
            float up[MC][4], t0[MC][4];
#pragma unroll
            for (int ch = 0; ch < MC; ++ch) {
                const float4 em = sE[sm][ch][lane_id], e0 = sE[s0][ch][lane_id];
                t0[ch][0] = e0.x; t0[ch][1] = e0.y; t0[ch][2] = e0.z; t0[ch][3] = e0.w;
                up[ch][0] = up3(em.x, e0.x, Ep[ch][0]);
                up[ch][1] = up3(em.y, e0.y, Ep[ch][1]);
                up[ch][2] = up3(em.z, e0.z, Ep[ch][2]);
                up[ch][3] = up3(em.w, e0.w, Ep[ch][3]);
            }
            float* f = a.fout ? a.fout + (((size_t)lane * a.h0 + 2 * j) * a.w0 + gx) * C : nullptr;
            egress_convert(a, pq, f, gx, in0, up);
            if (two) {
#pragma unroll
                for (int ch = 0; ch < MC; ++ch)
#pragma unroll
                    for (int i = 0; i < 4; ++i) up[ch][i] = up2(t0[ch][i], Ep[ch][i]);
                egress_convert(a, pq + a.out_step, f ? f + (size_t)a.w0 * C : nullptr, gx, in1, up);
            }
        }
        pq += 2 * a.out_step;
        const int t = sm; sm = s0; s0 = sp; sp = t;
    }
}

__global__ void k_copy(float* __restrict__ dst, const float* __restrict__ src, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

inline unsigned cdiv(int a, int b) { return (unsigned)((a + b - 1) / b); }

}  // namespace

// cuTensorMapEncodeTiled, resolved through the runtime so the library needs no link-time libcuda; thread-safe
// (several handles may be created from different threads: live chain + exporter)
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TensorMapEncodeFn tensor_map_encoder() {
    static const TensorMapEncodeFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || !p) {
            cudaGetLastError();
            p = nullptr;
        }
        return reinterpret_cast<TensorMapEncodeFn>(p);
    }();
    return fn;
}

// Encodes a 3-D tiled tensor map {w, h, planes} over pitched f32 planes with a box of box_w x box_h x 1 elements.
bool make_tensor_map_box(void* out_map, const float* base, const Level& l, int planes, int box_w, int box_h) {
    const TensorMapEncodeFn encode = tensor_map_encoder();
    if (!encode) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)l.w, (cuuint64_t)l.h, (cuuint64_t)planes};
    const cuuint64_t strides[2] = {(cuuint64_t)l.pitch * sizeof(float), (cuuint64_t)l.plane * sizeof(float)};
    const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    const CUresult r = encode(reinterpret_cast<CUtensorMap*>(out_map), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base),
                              dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

// the level kernel's boxes: input window (72 x 39, origin x0-4, y0-4) or state tile (64 x 32, origin x0, y0)
bool make_level_tensor_map(void* out_map, const float* base, const Level& l, int planes, bool state_tile) {
    return make_tensor_map_box(out_map, base, l, planes, state_tile ? TW : GW, state_tile ? TH : GH);
}

cudaError_t launch_lab16(const FrameIO& io, const DeviceTables& tb, int16_t* lab, int pitch16, size_t plane16,
                         cudaStream_t s, float* l_f32, int l_pitch, size_t l_plane) {
    const int aligned = (reinterpret_cast<uintptr_t>(io.in) % 4 == 0) && (io.in_step % 4 == 0) && (io.in_lane_stride % 4 == 0);
    dim3 grid(cdiv(cdiv(io.w, 4), 256), io.h, io.lanes);
    k_lab16<<<grid, 256, 0, s>>>(io.in, io.in_step, io.in_lane_stride, io.w, io.h, tb.lab_lut, lab, pitch16, plane16, aligned, l_f32, l_pitch, l_plane);
    return cudaGetLastError();
}

cudaError_t launch_ingest_lab(const FrameIO& io, const DeviceTables& tb, int16_t* lab, int pitch16, size_t plane16,
                              float* g1, const Level& l1, cudaStream_t s, int warps) {
    IngestArgs a;
    a.in = io.in; a.in_step = io.in_step; a.in_lane_stride = io.in_lane_stride;
    a.w = io.w; a.h = io.h;
    a.aligned = (reinterpret_cast<uintptr_t>(io.in) % 4 == 0) && (io.in_step % 4 == 0) && (io.in_lane_stride % 4 == 0);
    a.lut = tb.lab_lut; a.lab = lab; a.pitch16 = pitch16; a.plane16 = plane16; a.g1 = g1; a.l1 = l1;
    if (warps != 2 && warps != 4) warps = 1;
    dim3 grid(cdiv(io.w, DS_COLS), cdiv(l1.h, IG_ROWS * warps), io.lanes);
    if (warps == 4) k_ingest_lab<4><<<grid, 128, 0, s>>>(a);
    else if (warps == 2) k_ingest_lab<2><<<grid, 64, 0, s>>>(a);
    else k_ingest_lab<1><<<grid, 32, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_level(const LevelArgs& a, cudaStream_t s) {
    LevelKArgs k;
    k.g = a.g; k.in_plane = a.in_plane; k.in_row = a.in_row; k.channels = a.channels;
    for (int i = 0; i < 3; ++i) { k.sc[i] = a.sc[i]; k.of[i] = a.of[i]; }
    k.lf = a.lf; k.lc = a.lc; k.g_next = a.g_next; k.hi = a.hi; k.lo = a.lo; k.m = a.m;
    k.first = a.first; k.band = a.band;
    k.c_hi = a.c_hi; k.omc_hi = a.one_minus_c_hi; k.c_lo = a.c_lo; k.omc_lo = a.one_minus_c_lo;
    k.gain = a.gain;
    k.in_vec_ok = a.in_kind == IN_U8 ? ((reinterpret_cast<uintptr_t>(a.g) % 4 == 0) && (a.in_row % 4 == 0) && (a.in_plane % 4 == 0)) : 1;
    dim3 grid(cdiv(a.lf.w, TW), cdiv(a.lf.h, TH), a.planes);
    static const CUtensorMap dummy{};
    const CUtensorMap* tg = reinterpret_cast<const CUtensorMap*>(a.tmap);
    if (a.in_kind == IN_F32 && tg && a.tmap_hi && a.tmap_lo)
        k_level<IN_F32, true, true><<<grid, 256, 0, s>>>(k, *tg, *reinterpret_cast<const CUtensorMap*>(a.tmap_hi),
                                                          *reinterpret_cast<const CUtensorMap*>(a.tmap_lo));
    else if (a.in_kind == IN_F32 && tg) k_level<IN_F32, true, false><<<grid, 256, 0, s>>>(k, *tg, dummy, dummy);
    else if (a.in_kind == IN_F32) k_level<IN_F32, false, false><<<grid, 256, 0, s>>>(k, dummy, dummy, dummy);
    else if (a.in_kind == IN_LAB16) k_level<IN_LAB16, false, false><<<grid, 256, 0, s>>>(k, dummy, dummy, dummy);
    else k_level<IN_U8, false, false><<<grid, 256, 0, s>>>(k, dummy, dummy, dummy);
    return cudaGetLastError();
}

cudaError_t launch_down(const LevelArgs& a, cudaStream_t s) {
    DownArgs k;
    k.g = a.g; k.in_plane = a.in_plane; k.in_row = a.in_row; k.channels = a.channels;
    for (int i = 0; i < 3; ++i) { k.sc[i] = a.sc[i]; k.of[i] = a.of[i]; }
    k.lf = a.lf; k.lc = a.lc; k.g_next = a.g_next;
    k.in_vec_ok = a.in_kind == IN_U8 ? ((reinterpret_cast<uintptr_t>(a.g) % 4 == 0) && (a.in_row % 4 == 0) && (a.in_plane % 4 == 0)) : 1;
    dim3 grid(cdiv(a.lf.w, DS_COLS), cdiv(a.lc.h, DS_ROWS * DS_WARPS), a.planes);
    if (a.in_kind == IN_F32) k_down_strip<IN_F32><<<grid, 32 * DS_WARPS, 0, s>>>(k);
    else if (a.in_kind == IN_LAB16) k_down_strip<IN_LAB16><<<grid, 32 * DS_WARPS, 0, s>>>(k);
    else k_down_strip<IN_U8><<<grid, 32 * DS_WARPS, 0, s>>>(k);
    return cudaGetLastError();
}

cudaError_t launch_collapse(const Level& lf, const Level& lc, const BandSrc& fine, const BandSrc& coarse, float* out, int planes,
                            cudaStream_t s, int plane_step) {
    dim3 grid(cdiv(lf.w, TW), cdiv(lf.h, TH), planes / plane_step);
    k_collapse<<<grid, 256, 0, s>>>(lf, lc, fine, coarse, out, plane_step);
    return cudaGetLastError();
}

cudaError_t launch_egress(const FrameIO& io, const DeviceTables& tb, const int16_t* lab, int pitch16, size_t plane16,
                          const BandSrc& m1, const Level& l1, const BandSrc& c2, const Level& l2, float chroma,
                          float* fout, cudaStream_t s, int strip, int motion_channels) {
    EgressArgs a;
    a.in = io.in; a.in_step = io.in_step; a.in_lane_stride = io.in_lane_stride;
    a.lab = lab; a.pitch16 = pitch16; a.plane16 = plane16;
    a.out = io.out; a.out_step = io.out_step; a.out_lane_stride = io.out_lane_stride;
    a.w0 = io.w; a.h0 = io.h;
    a.gtab = tb.inv_gamma; a.coeffs = tb.inv_coeffs;
    a.m1 = m1; a.l1 = l1; a.c2 = c2; a.l2 = l2; a.chroma = chroma; a.fout = fout;
    if (strip) {
        dim3 grid(cdiv(io.w, DS_COLS), cdiv(io.h, EG_ROWS), io.lanes);
        // the register cap (resident warps per SM) of the three-channel kernel is an A/B knob: 16 -> <= 128 registers,
        // 20 -> 96, 24 -> 80.  The L-only kernel (chroma 0) has one cap, 24, chosen on a B200 (DESIGN §4).
        if (io.channels != 3) k_egress_strip<1, 1, 24><<<grid, 32, 0, s>>>(a);
        else if (motion_channels == 1) k_egress_strip<3, 1, 24><<<grid, 32, 0, s>>>(a);
        else if (strip == 16) k_egress_strip<3, 3, 16><<<grid, 32, 0, s>>>(a);
        else if (strip == 24) k_egress_strip<3, 3, 24><<<grid, 32, 0, s>>>(a);
        else k_egress_strip<3, 3, 20><<<grid, 32, 0, s>>>(a);
    } else {
        dim3 grid(cdiv(io.w, TW), cdiv(io.h, TH), io.lanes);
        if (io.channels != 3) k_egress<1, 1><<<grid, 256, 0, s>>>(a);
        else if (motion_channels == 1) k_egress<3, 1><<<grid, 256, 0, s>>>(a);
        else k_egress<3, 3><<<grid, 256, 0, s>>>(a);
    }
    return cudaGetLastError();
}

cudaError_t launch_copy_planes(float* dst, const float* src, size_t n, cudaStream_t s) {
    unsigned blocks = (unsigned)((n + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks == 0) blocks = 1;
    k_copy<<<blocks, 256, 0, s>>>(dst, src, n);
    return cudaGetLastError();
}

}  // namespace mc
