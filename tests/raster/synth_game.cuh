// TEST INFRASTRUCTURE. SynthOf<G>: a game whose frame is a synthetic scene (scene.h), with every render trait copied
// from the real game G, so that the rasteriser is instantiated exactly as the games compile it. build_frame uses only
// what the games use: tile_window, build_tile_layer and emit_post_blits with BlitReq::plain / rotated / rect.
#pragma once
#include "../../procgen2_b200/csrc/pg2_kernels.cuh"
#include "scene.h"

namespace pg2 {

// report[env * SC_REPORT + k]: 0 wide (as build_tile_layer left it), 1 npost, 2 reuse
constexpr int SC_REPORT = 4;

#define PG2_SYNTH_FIELDS(F)          \
    F(sc_scene, scene, 1)            \
    PG2_ENV_MAJOR(F)(int32_t, report, SC_REPORT)

PG2_DEFINE_STATE(SynthState, PG2_SYNTH_FIELDS)

template <class G>
struct SynthOf {
    using State = SynthState;
    static constexpr int MAX_POST = G::MAX_POST;
    static constexpr bool ROTATES = G::ROTATES;
    static constexpr int TILE_CLASSES = G::TILE_CLASSES;
    static constexpr int WIN_ROWS = G::WIN_ROWS;
    static constexpr int BLIT_UNROLL = G::BLIT_UNROLL;
    static constexpr bool HAS_TILES = G::HAS_TILES;
    static constexpr bool STATIC_VIEW = G::STATIC_VIEW;
    static constexpr int RENDER_MIN_CTAS = G::RENDER_MIN_CTAS;
    static constexpr int NUM_TEX = SC_NUM_TEX;
    static_assert(SC_NUM_TEX >= MAX_TILE_TEX, "tile texture ids are < MAX_TILE_TEX");

    static PG2_DEV int tile_class(uint32_t t) { return sc_tile_class((int)t, TILE_CLASSES); }

    template <class F>
    static PG2_DEV_NOINLINE void build_frame(const State& s, const CommonState& c, int env, F& f, const TexInfo* tex) {
        (void)c;
        const sc_scene& sc = s.scene[env];
        Camera cam{ sc.cam_x, sc.cam_y, __fdiv_rn(__fmul_rn(sc.cam_scale, f.view_w), 64.0f), f.view_w, f.view_h };
        int lx = 0, ly = 0, ux = -1, uy = -1;
        if (HAS_TILES) tile_window(cam, &lx, &ly, &ux, &uy);
        const int ncol = min(ux - lx + 1, MAX_WIN), nrow = min(uy - ly + 1, MAX_WIN);
        build_tile_layer(f, cam, tex, TILE_CLASSES, lx, ly, ncol, nrow, [](int cls) { return cls ? 16 : 0; },
                         [&](int x, int y) { const int t = sc_tile_at(&sc, x, y); return t == SC_NO_TILE ? (int)NO_TILE : t; },
                         sc.bg_tex, sc.bg_x, sc.bg_y, sc.bg_scale);
        emit_post_blits(f, tex, sc.npost, [&](int k, BlitReq& b, BlitRot& rot) {
            const sc_post& p = sc.post[k];
            if (p.mode == 1) b.plain(p.tex, p.x, p.y, cam, p.scale, p.alpha, p.flip != 0);
            else if (p.mode == 2) b.rotated(p.tex, p.x, p.y, cam, p.rotation, p.scale, p.alpha, &rot);
            else if (p.mode == 3) b.rect(p.tex, p.x, p.y, p.w, p.h, p.angle, &rot);
        });
        __syncthreads();   // f.npost and f.wide are complete
        if (threadIdx.x == 0) {
            int32_t* r = s.report + (size_t)env * SC_REPORT;
            r[0] = f.wide; r[1] = f.npost; r[2] = f.reuse;
        }
    }
};

}  // namespace pg2
