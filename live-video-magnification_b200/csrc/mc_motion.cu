// Motion (Laplace) per-frame driver — device twin of magcore::magnifyMotion
// (reference src/processing/magnification/MagnifyCore.hpp:83-160).
#include <algorithm>
#include <cstring>

#include "mc_modes.h"

namespace mc {

cudaError_t DeviceArena::alloc(float** p, size_t floats) {
    void* v = nullptr;
    cudaError_t e = alloc_bytes(&v, floats * sizeof(float));
    *p = (float*)v;
    return e;
}
cudaError_t DeviceArena::alloc_bytes(void** p, size_t bytes) {
    *p = nullptr;
    cudaError_t e = cudaMalloc(p, bytes ? bytes : 4);
    if (e == cudaSuccess) blocks.push_back(*p);
    return e;
}
void DeviceArena::free_block(void* p) {
    for (size_t i = 0; i < blocks.size(); ++i)
        if (blocks[i] == p) {
            cudaFree(p);
            blocks.erase(blocks.begin() + (long)i);
            return;
        }
}
void DeviceArena::release() {
    for (void* b : blocks) cudaFree(b);
    blocks.clear();
}

void MotionMode::drop_groups() {
    for (Group& g : groups) {
        if (g.stream) { cudaStreamSynchronize(g.stream); cudaStreamDestroy(g.stream); }
        if (g.done) cudaEventDestroy(g.done);
    }
    groups.clear();
    if (ev_fork) { cudaEventDestroy(ev_fork); ev_fork = nullptr; }
}

void MotionMode::reset() {
    drop_groups();
    arena.release();
    lv.clear(); G.clear(); hi.clear(); lo.clear(); M.clear();
    lab16 = nullptr;
    allocated = false;
    empty = true;
}

// (Re)builds the lane groups — their streams, events and TMA descriptors — over the existing buffers; the temporal state
// is untouched, so the option can change between frames (profile_kernels forces one group).
mc_status MotionMode::make_groups(const ModeCtx& ctx) {
    // lane groups: automatic = two chains once each has >= 8 streams.  B200, 32 lanes x 1080p: 1 group 27.9 k frames/s,
    // 2 groups 29.2 k, 4 groups 29.0 k, 8 groups 28.6 k; serialising the same stage of consecutive groups with events
    // (so that different stages overlap by construction) was slower than one chain (24.1 k): the stages contend for the
    // same L1 data pipe, so co-residency buys little beyond filling each other's tails.
    drop_groups();
    groups_req = ctx.lane_groups;
    int ng = groups_req > 0 ? groups_req : std::min(2, lanes / 8);
    ng = std::max(1, std::min(ng, lanes));
    groups.assign((size_t)ng, Group{});
    for (int g = 0; g < ng; ++g) {
        Group& grp = groups[(size_t)g];
        grp.lane0 = (int)((long long)lanes * g / ng);
        grp.lanes = (int)((long long)lanes * (g + 1) / ng) - grp.lane0;
        if (ng > 1) {
            MCK(cudaStreamCreateWithFlags(&grp.stream, cudaStreamNonBlocking));
            MCK(cudaEventCreateWithFlags(&grp.done, cudaEventDisableTiming));
        }
        // TMA descriptors for the f32 inputs and the state planes of the fused level kernels, over this group's planes
        const size_t p0 = (size_t)grp.lane0 * channels;
        const int gp = grp.lanes * channels;
        grp.tmaps.assign((size_t)levels + 1, TensorMapStorage{});
        grp.tmaps_hi.assign((size_t)levels + 1, TensorMapStorage{});
        grp.tmaps_lo.assign((size_t)levels + 1, TensorMapStorage{});
        grp.tmap_valid.assign((size_t)levels + 1, 0);
        for (int l = 1; l < levels; ++l) {
            const Level& L = lv[(size_t)l];
            grp.tmap_valid[(size_t)l] = make_level_tensor_map(&grp.tmaps[(size_t)l], G[(size_t)l] + p0 * L.plane, L, gp) &&
                                        make_level_tensor_map(&grp.tmaps_hi[(size_t)l], hi[(size_t)l] + p0 * L.plane, L, gp, true) &&
                                        make_level_tensor_map(&grp.tmaps_lo[(size_t)l], lo[(size_t)l] + p0 * L.plane, L, gp, true) ? 1 : 0;
        }
    }
    if (ng > 1) MCK(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
    return MC_OK;
}

mc_status MotionMode::allocate(const ModeCtx& ctx, const FrameIO& io, int nlevels) {
    reset();
    levels = nlevels; channels = io.channels; w = io.w; h = io.h;
    faithful = ctx.faithful0;
    from_state = ctx.band_from_state;
    const size_t planes = (size_t)lanes * channels;
    lv.resize((size_t)levels + 1);
    int cw = w, ch = h;
    for (int l = 0; l <= levels; ++l) {
        lv[(size_t)l] = make_level(cw, ch);
        cw = (cw + 1) / 2;
        ch = (ch + 1) / 2;
    }
    G.assign((size_t)levels + 1, nullptr);
    hi.assign((size_t)levels + 1, nullptr);
    lo.assign((size_t)levels + 1, nullptr);
    M.assign((size_t)levels + 1, nullptr);
    for (int l = 0; l <= levels; ++l) {
        const size_t n = planes * lv[(size_t)l].plane;
        const bool band_level = l < levels;                       // bands 0..levels-1, residual = levels
        const bool live = band_level && l >= 1;                   // bands whose gain can be non-zero
        if (l >= 1) MCK(arena.alloc(&G[(size_t)l], n));
        if (live || faithful) {
            MCK(arena.alloc(&hi[(size_t)l], n));
            MCK(arena.alloc(&lo[(size_t)l], n));
        }
        // M_l: the amplified band of level l, overwritten by the collapsed cur_l.  With band_from_state the bands are
        // rebuilt from hi/lo by their consumers and only cur_2 .. cur_{levels-2} are materialised.
        if (live && (!from_state || (l >= 2 && l <= levels - 2))) MCK(arena.alloc(&M[(size_t)l], n));
    }
    if (channels == 3) {
        pitch16 = round_up(w, 64);
        plane16 = (size_t)h * pitch16;
        void* p = nullptr;
        MCK(arena.alloc_bytes(&p, planes * plane16 * sizeof(int16_t)));
        lab16 = (int16_t*)p;
    }
    MCK_ST(make_groups(ctx));
    allocated = true;
    return MC_OK;
}

mc_status MotionMode::process(const ModeCtx& ctx, const FrameIO& io, const mc_params& p, int nlevels, int* produced) {
    if (!allocated || faithful != ctx.faithful0 || from_state != ctx.band_from_state) {
        mc_status st = allocate(ctx, io, nlevels);
        if (st != MC_OK) return st;
    } else if (groups_req != ctx.lane_groups) {
        mc_status st = make_groups(ctx);
        if (st != MC_OK) return st;
    }
    const bool first = empty;  // MagnifyCore.hpp:98
    motion_gains(p.amplification, p.coWavelength, levels, w, h, gains);
    double c_lo = p.coLow, c_hi = p.coHigh;
    if (c_lo == 0) c_lo = 0.01;  // TemporalFilter.cpp:11-12

    if (groups.size() == 1) {
        const mc_status st = run_group(ctx, io, p, groups[0], first, c_lo, c_hi);
        if (st != MC_OK) return st;
    } else {
        // fork: every group's chain starts after whatever the caller queued on the handle's stream (the frame upload),
        // join: the handle's stream continues after all of them (the download / the caller's next use of `out`)
        MCK(cudaEventRecord(ev_fork, ctx.stream));
        for (Group& g : groups) {
            MCK(cudaStreamWaitEvent(g.stream, ev_fork, 0));
            ModeCtx gctx = ctx;
            gctx.stream = g.stream;
            const mc_status st = run_group(gctx, io, p, g, first, c_lo, c_hi);
            if (st != MC_OK) return st;
            MCK(cudaEventRecord(g.done, g.stream));
            MCK(cudaStreamWaitEvent(ctx.stream, g.done, 0));
        }
    }
    if (ctx.analysis_only && !first) {   // state-carry pass: the temporal state is up to date, no frame is produced
        *produced = 0;
        return MC_OK;
    }
    empty = false;
    *produced = 1;
    return MC_OK;
}

// One group's launch set for one frame: lanes [g.lane0, g.lane0 + g.lanes) on ctx.stream.
mc_status MotionMode::run_group(const ModeCtx& ctx, const FrameIO& io_all, const mc_params& p, Group& g, bool first, double c_lo, double c_hi) {
    FrameIO io = io_all;
    io.in = io_all.in + (size_t)g.lane0 * io_all.in_lane_stride;
    io.out = io_all.out + (size_t)g.lane0 * io_all.out_lane_stride;
    io.lanes = g.lanes;
    const int planes = g.lanes * channels;
    const size_t p0 = (size_t)g.lane0 * channels;
    auto off = [&](float* base, int l) { return base ? base + p0 * lv[(size_t)l].plane : nullptr; };
    int16_t* lab = lab16 ? lab16 + p0 * plane16 : nullptr;
    float* fout = ctx.float_out ? ctx.float_out + (size_t)g.lane0 * w * h * channels : nullptr;

    // ingest: u8 BGR -> Lab16 planes (gray frames are read directly by the level-0 kernel)
    // (production path, >= 2 levels: one fused kernel also builds G1; otherwise Lab16 alone)
    const bool fused_ingest = channels == 3 && !faithful && levels >= 2;
    if (fused_ingest) LAUNCH("ingest_lab", 0, launch_ingest_lab(io, *ctx.tables, lab, pitch16, plane16, off(G[1], 1), lv[1], ctx.stream, ctx.ingest_warps));
    else if (channels == 3) LAUNCH("lab16", 0, launch_lab16(io, *ctx.tables, lab, pitch16, plane16, ctx.stream));

    // analysis: one fused kernel per level (level 0 only builds G1 unless the faithful option is on)
    const int l_begin = fused_ingest ? 1 : ((levels >= 2 || faithful) ? 0 : levels);
    for (int l = l_begin; l < levels; ++l) {
        LevelArgs a;
        if (l == 0) {
            if (channels == 3) {
                a.in_kind = 1; a.g = lab; a.in_plane = plane16; a.in_row = pitch16;
                a.sc[0] = 100.0f / 16384.0f; a.of[0] = 0.0f;
                a.sc[1] = a.sc[2] = 1.0f / 64.0f; a.of[1] = a.of[2] = -128.0f;
            } else {
                a.in_kind = 2; a.g = io.in; a.in_plane = io.in_lane_stride; a.in_row = (int)io.in_step;
                a.sc[0] = 0.003921568859368563f;
            }
        } else {
            a.in_kind = 0; a.g = off(G[(size_t)l], l); a.in_plane = lv[(size_t)l].plane; a.in_row = lv[(size_t)l].pitch;
            if (g.tmap_valid[(size_t)l] && ctx.use_tma) {
                a.tmap = &g.tmaps[(size_t)l];
                if (ctx.prefetch_state) { a.tmap_hi = &g.tmaps_hi[(size_t)l]; a.tmap_lo = &g.tmaps_lo[(size_t)l]; }
            }
        }
        a.channels = channels;
        a.lf = lv[(size_t)l]; a.lc = lv[(size_t)l + 1];
        a.g_next = off(G[(size_t)l + 1], l + 1);
        a.hi = off(hi[(size_t)l], l); a.lo = off(lo[(size_t)l], l);
        a.m = (first || from_state) ? nullptr : off(M[(size_t)l], l);
        a.planes = planes;
        a.first = first ? 1 : 0;
        a.band = (l >= 1 || faithful) ? 1 : 0;
        a.c_hi = c_hi; a.one_minus_c_hi = 1 - c_hi; a.c_lo = c_lo; a.one_minus_c_lo = 1 - c_lo;
        a.gain = gains[(size_t)l];
        if (a.band) LAUNCH("level", l, launch_level(a, ctx.stream));
        else LAUNCH("down", l, launch_down(a, ctx.stream));
    }
    if (first && faithful)  // st.lowpassHi/Lo[levels] = residual (MagnifyCore.hpp:100-101)
    {
        const size_t n = (size_t)planes * lv[(size_t)levels].plane;
        LAUNCH("copy", levels, launch_copy_planes(off(hi[(size_t)levels], levels), off(G[(size_t)levels], levels), n, ctx.stream));
        LAUNCH("copy", levels, launch_copy_planes(off(lo[(size_t)levels], levels), off(G[(size_t)levels], levels), n, ctx.stream));
    }
    if (ctx.analysis_only && !first) return MC_OK;
    // chroma 0 multiplies the a and b planes of the motion image by 0 before input + motion (MagnifyCore.hpp:140-148),
    // which leaves the input's a and b exactly as they are (DESIGN §4): the synthesis then runs on the L planes alone.
    // The a and b state above keeps evolving, so a later frame with chroma != 0 is unaffected.  NaN compares unequal.
    const int motion_channels = (channels == 3 && (float)p.chromAttenuation == 0.0f) ? 1 : channels;
    BandSrc m1, c2;
    if (!first && levels >= 2) {
        // synthesis: residual and finest band are zero (MagnifyCore.hpp:130-131), so the collapse starts from
        // band levels-1 (cur_{levels-1} = 0 + m_{levels-1}); levels 1 and 0 are folded into egress.
        auto band = [&](int l) {
            return from_state ? BandSrc{off(hi[(size_t)l], l), off(lo[(size_t)l], l), gains[(size_t)l]} : BandSrc{off(M[(size_t)l], l), nullptr, 1.0f};
        };
        auto cur = [&](int l) { return l == levels - 1 ? band(l) : BandSrc{off(M[(size_t)l], l), nullptr, 1.0f}; };
        for (int l = levels - 2; l >= 2; --l)
            LAUNCH("collapse", l, launch_collapse(lv[(size_t)l], lv[(size_t)l + 1], band(l), cur(l + 1), off(M[(size_t)l], l), planes, ctx.stream,
                                                  channels / motion_channels));
        m1 = band(1);
        if (levels >= 3) c2 = cur(2);
    }
    const Level& l1 = lv[levels >= 1 ? 1 : 0];
    const Level& l2 = lv[levels >= 2 ? 2 : 0];
    LAUNCH("egress", 0, launch_egress(io, *ctx.tables, lab, pitch16, plane16, m1, l1, c2, l2, (float)p.chromAttenuation, fout,
                                      ctx.stream, ctx.egress_strip, motion_channels));
    return MC_OK;
}

void MotionMode::find_state(const char* name, int level, StateRef& out) {
    out = StateRef{};
    if (!allocated || empty || level < 0 || level > levels) return;
    float* p = nullptr;
    if (!std::strcmp(name, "lowpassHi")) p = hi[(size_t)level];
    else if (!std::strcmp(name, "lowpassLo")) p = lo[(size_t)level];
    if (!p) return;
    const Level& l = lv[(size_t)level];
    out.ptr = p; out.rows = l.h; out.cols = l.w; out.channels = channels; out.pitch = l.pitch; out.plane_stride = l.plane;
}

}  // namespace mc
