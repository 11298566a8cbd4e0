// Internal interfaces between the handle (mc_core.cu), the tables (mc_tables.cpp) and the kernel
// launchers (mc_laplace.cu, mc_color.cu, mc_riesz.cu).  Not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "mc_math.cuh"

namespace mc {

// Geometry of one pyramid level; planes are f32 [plane][h][pitch] with pitch % 32 == 0.
struct Level {
    int w = 0, h = 0, pitch = 0;
    size_t plane = 0;  // floats per plane = h * pitch
};

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

inline Level make_level(int w, int h) {
    Level l;
    l.w = w; l.h = h; l.pitch = round_up(w, 32); l.plane = (size_t)l.h * l.pitch;
    return l;
}

// Device constant tables shared by every handle on a device (built once per device).
struct DeviceTables {
    LabLutCell* lab_lut = nullptr;   // [34][33][33] cells (mc_math.cuh)
    float4* inv_gamma = nullptr;      // [1024] spline coefficients {f, b, c, d}
    LabInvCoeffs inv_coeffs{};
};

// mc_tables.cpp ------------------------------------------------------------------------------
void build_lab_lut_cells(std::vector<LabLutCell>& out);          // from the embedded int16 table
void build_inv_gamma_spline(std::vector<float4>& out);             // OpenCV sRGBInvGammaTab
void build_lab_inv_coeffs(LabInvCoeffs& out);
int calculate_max_levels(int w, int h);
int optimal_buffer_size(int fps);
void butterworth(unsigned order, double wn, std::vector<double>& a, std::vector<double>& b);
void motion_gains(double amplification, double coWavelength, int levels, int w, int h, std::vector<float>& gains);
void gaussian_kernel_13_3(float taps[13]);
void build_area_tab(int ssize, int dsize, double scale, std::vector<AreaTap>& tab, std::vector<int>& ofs);
void preprocess_roi(int cols, int rows, bool enabled, float rx, float ry, float rw, float rh, int& x, int& y, int& w, int& h);

// ------------------------------------------------------------------------------------------------
// Laplace launchers (mc_laplace.cu).  All take the handle's stream; every call is one kernel launch
// and returns the launch's cudaError_t (cudaGetLastError()).
// ------------------------------------------------------------------------------------------------
struct FrameIO {
    const uint8_t* in = nullptr;   // [lanes][h][in_step]
    size_t in_step = 0, in_lane_stride = 0;
    uint8_t* out = nullptr;
    size_t out_step = 0, out_lane_stride = 0;
    int w = 0, h = 0, channels = 0, lanes = 0;
};

// u8 BGR frame -> Lab int16 planes [lanes*3][h][pitch16] (exact OpenCV LUT values, SURVEY A.3)
// (l_f32 != null: also the L plane as f32 [lanes][h][l_pitch] — Phase's input)
cudaError_t launch_lab16(const FrameIO& io, const DeviceTables& tb, int16_t* lab, int pitch16, size_t plane16,
                         cudaStream_t s, float* l_f32 = nullptr, int l_pitch = 0, size_t l_plane = 0);

// fused ingest of the production path: u8 BGR -> Lab16 planes + G1 = pyrDown(Lab) (MagnifyCore.hpp:87-96, level 0)
cudaError_t launch_ingest_lab(const FrameIO& io, const DeviceTables& tb, int16_t* lab, int pitch16, size_t plane16,
                              float* g1, const Level& l1, cudaStream_t s, int warps_per_cta = 1);

struct LevelArgs {
    int in_kind = 0;           // 0: f32 planes, 1: Lab int16 planes, 2: u8 gray frame
    const void* g = nullptr;   // input planes of this level (fine)
    size_t in_plane = 0;       // elements between planes
    int in_row = 0;            // elements between rows
    int channels = 1;
    float sc[3] = {1, 1, 1}, of[3] = {0, 0, 0};   // value = fma(raw, sc[ch], of[ch]) for kinds 1, 2
    Level lf, lc;              // this level (fine) and the next (coarse)
    float* g_next = nullptr;   // G_{l+1} planes (written)
    float* hi = nullptr; float* lo = nullptr;     // state planes of this level
    float* m = nullptr;        // gain * (hi - lo), may be null
    int planes = 0;
    int first = 0;             // 1: hi = lo = band (MagnifyCore.hpp:98-103)
    int band = 1;              // 0: only pyrDown (the level-0 band never reaches the output)
    double c_hi = 0, one_minus_c_hi = 0, c_lo = 0, one_minus_c_lo = 0;
    float gain = 0;
    const void* tmap = nullptr;   // CUtensorMap of the f32 input planes (TMA-staged tile) or null
    const void* tmap_hi = nullptr, *tmap_lo = nullptr;   // CUtensorMaps of the state planes: prefetch their tiles too
};
// 128-byte opaque CUtensorMap storage + encoder for the level kernel's (72 x 39 x 1) box
struct alignas(64) TensorMapStorage { unsigned char bytes[128]; };
bool make_level_tensor_map(void* out_map, const float* base, const Level& l, int planes, bool state_tile = false);
// general form: box of box_w x box_h x 1 f32 elements (row bytes must be a multiple of 16)
bool make_tensor_map_box(void* out_map, const float* base, const Level& l, int planes, int box_w, int box_h);
// fused per level: pyrDown + pyrUp + subtract + dual-EMA update + gain (SpatialFilter.cpp:25-38,
// TemporalFilter.cpp:9-22, MagnifyCore.hpp:127-134)
cudaError_t launch_level(const LevelArgs& a, cudaStream_t s);
// pure pyrDown of `a.g` into `a.g_next` (register/shuffle strip kernel; used when a.band == 0)
cudaError_t launch_down(const LevelArgs& a, cudaStream_t s);

// Where the synthesis kernels find a band: either a stored plane set (b == nullptr: value = a[i]) or the two
// temporal-filter state plane sets of that level, from which the amplified band-pass is rebuilt on the fly as
// gain * (a[i] - b[i]) = gain * (lowpassHi - lowpassLo) (TemporalFilter.cpp:21, MagnifyCore.hpp:127-134).
struct BandSrc {
    const float* a = nullptr;
    const float* b = nullptr;
    float gain = 1.0f;
};

// out_l = pyrUp(coarse) + fine (SpatialFilter.cpp:52-61); `out` may be the stored fine plane itself (in place).
// plane_step: 1 collapses every one of `planes` planes, 3 only the first (L) plane of each of planes / 3 lanes.
cudaError_t launch_collapse(const Level& lf, const Level& lc, const BandSrc& fine, const BandSrc& coarse, float* out, int planes,
                            cudaStream_t s, int plane_step = 1);

// out = convert(input + chroma * pyrUp(pyrUp(c2) + m1)) (MagnifyCore.hpp:136-158).
// m1.a == nullptr: no motion; c2.a == nullptr: cur_1 = m1.  C == 3 reads `lab`, C == 1 reads io.in.
// motion_channels == 1 with C == 3 (chroma == 0): only the L planes of m1 / c2 are read, a and b pass through unchanged.
cudaError_t launch_egress(const FrameIO& io, const DeviceTables& tb, const int16_t* lab, int pitch16, size_t plane16,
                          const BandSrc& m1, const Level& l1, const BandSrc& c2, const Level& l2, float chroma,
                          float* float_out_or_null, cudaStream_t s, int strip = 20, int motion_channels = 3);

// PreprocessProcessor + GrayscaleProcessor on the device (mc_preprocess.cu)
cudaError_t launch_preprocess(const uint8_t* src_roi, size_t step, int cn, int sw, int sh, int dw, int dh, bool copy_only,
                              const AreaTap* xtab, const int* xofs, const AreaTap* ytab, const int* yofs, uint8_t* dst,
                              uint8_t* gray, cudaStream_t s);

// plane copy helpers
cudaError_t launch_copy_planes(float* dst, const float* src, size_t n, cudaStream_t s);

}  // namespace mc
