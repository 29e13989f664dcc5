// Shared device-side building blocks of the batched Procgen2 engine (B200 / sm_100a).
// Everything here restates arithmetic of the reference's copy-pasted mini engine, which is
// byte-identical across the seven games (SURVEY.md §2.2): helpers.cpp (AABB maths),
// renderer.cpp (world->screen transform of one blit). Float code is compiled with
// -fmad=false so that every operation rounds exactly like the x86-64 baseline build (Q14);
// the explicit __f*_rn intrinsics below additionally forbid contraction where it matters most.
#pragma once
#include <stdint.h>
#include "pg2_platform.cuh"
#include "pg2_types.h"

namespace pg2 {

constexpr float UNIT_TO_PIXELS = 16.0f;          // helpers.h:8
constexpr float PIXELS_TO_UNIT = 1.0f / 16.0f;   // helpers.h:9
constexpr int OBS_W = 64, OBS_H = 64, OBS_BYTES = 64 * 64 * 3;

// How ONE environment's cenv_step is spread over threads: nlanes == 1 (one thread owns the environment:
// thread-per-env mapping, host-sim) or nlanes == WARP_LANES (a whole warp owns it: per-entity loops are strided
// over the lanes, everything else is computed redundantly by all lanes, which therefore stay converged).
// nlanes may also be a PART of a warp (8 or 16 lanes, `mask` = the group's lanes): several environments share a warp, each
// with its own lane group — the uniform code then issues once for all of them.
struct StepCtx {
    int lane, nlanes;
    uint32_t mask = 0xffffffffu;
    PG2_DEV bool any(bool p) const { return nlanes == 1 ? p : group_any(mask, p); }
    PG2_DEV int sum(int v) const { return nlanes == 1 ? v : group_sum(mask, v); }
    PG2_DEV uint64_t or64(uint64_t v) const { return nlanes == 1 ? v : (uint64_t)group_or(mask, (uint32_t)v) | (uint64_t)group_or(mask, (uint32_t)(v >> 32)) << 32; }
    PG2_DEV void sync() const { if (nlanes != 1) group_sync(mask); }
    PG2_DEV bool leader() const { return lane == 0; }
};

struct Rect { float x, y, w, h; };
struct Vec2 { float x, y; };

// x86-64 `cvttss2si` semantics for float->int casts (NaN / out of range -> INT_MIN);
// CUDA's own cast saturates instead, which would diverge on degenerate blit rectangles.
PG2_DEV int f2i(float f) {
    return (f > -2147483904.0f && f < 2147483648.0f) ? (int)f : (int)0x80000000;
}
PG2_DEV int d2i(double f) {
    return (f > -2147483649.0 && f < 2147483648.0) ? (int)f : (int)0x80000000;
}

// helpers.cpp:40-46
PG2_DEV bool check_collision(const Rect& a, const Rect& b) {
    return (a.x < (b.x + b.w) && (a.x + a.w) > b.x) && (a.y < (b.y + b.h) && (a.y + a.h) > b.y);
}

// helpers.cpp:48-108 (raylib-style overlap rectangle)
PG2_DEV Rect get_collision_overlap(const Rect& r1, const Rect& r2) {
    Rect res{ 0.0f, 0.0f, 0.0f, 0.0f };
    if (check_collision(r1, r2)) {
        float dxx = fabsf(r1.x - r2.x);
        float dyy = fabsf(r1.y - r2.y);
        if (r1.x <= r2.x) {
            if (r1.y <= r2.y) { res.x = r2.x; res.y = r2.y; res.w = r1.w - dxx; res.h = r1.h - dyy; }
            else              { res.x = r2.x; res.y = r1.y; res.w = r1.w - dxx; res.h = r2.h - dyy; }
        } else {
            if (r1.y <= r2.y) { res.x = r1.x; res.y = r2.y; res.w = r2.w - dxx; res.h = r1.h - dyy; }
            else              { res.x = r1.x; res.y = r1.y; res.w = r2.w - dxx; res.h = r2.h - dyy; }
        }
        if (r1.w > r2.w) { if (res.w >= r2.w) res.w = r2.w; }
        else             { if (res.w >= r1.w) res.w = r1.w; }
        if (r1.h > r2.h) { if (res.h >= r2.h) res.h = r2.h; }
        else             { if (res.h >= r1.h) res.h = r1.h; }
    }
    return res;
}

// 16.16 source increment (sl << 16) / dl; a 32-bit divide whenever the numerator fits (always, for real textures).
PG2_DEV uint32_t fixed_inc(int sl, int dl) {
    return sl < 65536 ? ((uint32_t)sl << 16) / (uint32_t)dl : (uint32_t)(((uint64_t)sl << 16) / (uint64_t)dl);
}

// One axis of Renderer::render_texture (renderer.cpp:5-82). The reference treats x and y
// independently, so the crop/pad/compensate arithmetic is evaluated per axis; the same
// descriptor also serves whole tile columns / rows of the tile layer.
struct Axis {
    int d0, dlen;      // integer destination start / length (SDL truncates the float dst rect)
    int s0;            // first source texel after clipping the source rect to the texture
    uint32_t inc;      // 16.16 source increment per destination pixel
    int visible;       // 0 when culled or degenerate
};

// pos: world position in pixels, cam: camera position, cs: camera scale, size: screen size,
// tex_len: texture extent on this axis, scale: render scale, flip: mirror the source rect
// (horizontal flip only affects the x axis), y_axis selects the asymmetric cull test
// (renderer.cpp:14: `dst.x > size.x || dst.y >= size.y`).
PG2_DEV Axis make_axis_inl(float pos, float cam, float cs, float size, int tex_len, float scale, bool flip, bool y_axis) {
    Axis a; a.visible = 0; a.d0 = 0; a.dlen = 0; a.s0 = 0; a.inc = 0;
    float src0 = 0.0f, srcl = (float)tex_len;
    float dst0 = __fadd_rn(__fmul_rn(__fsub_rn(pos, cam), cs), __fmul_rn(size, 0.5f));
    float dstl = __fmul_rn(__fmul_rn((float)tex_len, scale), cs);
    if (y_axis ? (dst0 >= size) : (dst0 > size)) return a;
    if (__fadd_rn(dst0, dstl) < 0.0f) return a;
    if (dst0 < 0.0f) {
        float ratio = __fdiv_rn(-dst0, dstl);
        src0 = __fadd_rn(src0, __fmul_rn(srcl, ratio));
        srcl = __fsub_rn(srcl, src0);
        dstl = __fadd_rn(dstl, dst0);
        dst0 = 0.0f;
    }
    if (__fadd_rn(dst0, dstl) > size) {
        float ratio = __fdiv_rn(__fsub_rn(__fadd_rn(dst0, dstl), size), dstl);
        srcl = __fmul_rn(srcl, __fsub_rn(1.0f, ratio));
        dstl = __fsub_rn(size, dst0);
    }
    int padding = f2i(ceilf(__fdiv_rn(1.0f, __fmul_rn(scale, cs))));
    int si0 = f2i(floorf(src0));
    int sil = f2i(ceilf(srcl)) + padding;
    float offset = __fsub_rn(src0, (float)si0);
    float size_ratio = __fdiv_rn((float)sil, srcl);
    dstl = __fmul_rn(dstl, size_ratio);
    dst0 = __fsub_rn(dst0, __fmul_rn(offset, __fdiv_rn(dstl, srcl)));
    if (flip) si0 = tex_len - sil - si0;
    // SDL side (canonical rasteriser, oracle/raster.c): clip the source rect to the texture
    // in float, truncate both rects to int.
    float amin = (float)si0, amax = __fadd_rn((float)si0, (float)sil);
    if (amin < 0.0f) amin = 0.0f;
    if (amax > (float)tex_len) amax = (float)tex_len;
    int s0 = f2i(amin), sl = f2i(__fsub_rn(amax, amin));
    int d0 = f2i(dst0), dl = f2i(dstl);
    if (sl <= 0 || dl <= 0) return a;
    a.d0 = d0; a.dlen = dl; a.s0 = s0;
    a.inc = fixed_inc(sl, dl);
    a.visible = 1;
    return a;
}

PG2_TU_LOCAL PG2_DEV_CALL Axis make_axis(float pos, float cam, float cs, float size, int tex_len, float scale, bool flip, bool y_axis) {
    return make_axis_inl(pos, cam, cs, size, tex_len, scale, flip, y_axis);
}

// Both axes of Renderer::render_texture in one function body: the two chains are independent, so their long
// dependent float sequences interleave (twice the instruction-level parallelism of two make_axis calls).
PG2_TU_LOCAL PG2_DEV_CALL void make_axis_xy(float px, float py, float cam_x, float cam_y, float cs, float size_x, float size_y, int tex_w, int tex_h,
                                   float scale, bool flip_h, Axis* ax, Axis* ay) {
    *ax = make_axis_inl(px, cam_x, cs, size_x, tex_w, scale, flip_h, false);
    *ay = make_axis_inl(py, cam_y, cs, size_y, tex_h, scale, false, true);
}

// Axis of a blit whose float destination rect is given directly and whose source is the whole
// texture (Renderer::render_texture_rotated renderer.cpp:84-101, jumper HUD jumper.cpp:487-508).
PG2_DEV Axis make_axis_direct(float dst0, float dstl, int tex_len) {
    Axis a; a.visible = 0; a.s0 = 0; a.inc = 0;
    a.d0 = f2i(dst0); a.dlen = f2i(dstl);
    if (a.dlen <= 0 || tex_len <= 0) return a;
    a.inc = fixed_inc(tex_len, a.dlen);
    a.visible = 1;
    return a;
}

// A resolved blit: both axes + texture + modifiers. 52 bytes, lives in shared memory only.
struct Blit {
    Axis ax, ay;
    uint32_t tex_offset;
    uint16_t tex_w;
    uint8_t blend, alpha_mod, flip_h, rotated;
};

// SRC-over with SDL's classic integer arithmetic (oracle/raster.c blend_px).
PG2_DEV void blend_texel(uint32_t& r, uint32_t& g, uint32_t& b, uint32_t texel, uint32_t blend, uint32_t alpha_mod) {
    uint32_t tr = texel & 255u, tg = (texel >> 8) & 255u, tb = (texel >> 16) & 255u, ta = texel >> 24;
    if (!blend) { r = tr; g = tg; b = tb; return; }
    if (alpha_mod != 255u) ta = (ta * alpha_mod) / 255u;
    if (ta < 255u) { tr = (tr * ta) / 255u; tg = (tg * ta) / 255u; tb = (tb * ta) / 255u; }
    uint32_t ia = 255u - ta;
    r = tr + (ia * r) / 255u;
    g = tg + (ia * g) / 255u;
    b = tb + (ia * b) / 255u;
}

PG2_DEV int axis_sample(const Axis& a, int p, bool flip) {
    int i = p - a.d0;
    if (flip) i = a.dlen - 1 - i;
    return a.s0 + (int)((a.inc / 2u + (uint32_t)i * a.inc) >> 16);
}

}  // namespace pg2
