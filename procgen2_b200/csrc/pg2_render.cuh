// Observation rasteriser: one CTA renders one environment's 64x64x3 frame.
//
// Replaces render_game() (games/coinrun/coinrun.cpp:443-470 and its six siblings) together with
// the SDL3 software blits it issues (SDL_RenderTextureRotated, renderer.cpp:78/97) and the
// RGBA->RGB pack loop (coinrun.cpp:377-388). Draw order is the reference's painter's order:
//   clear(0,0,0) -> "pre" blit (background) -> tile layer (y-major, x-minor; tilemap.cpp:303-320)
//   -> "post" blits (particles, sprites, agent, HUD) in submission order.
//
// The frame is drawn in shared memory by row bands (8 bands x 8 rows, handed out to the CTA's warps), as RGBA words:
//   base pass   every thread owns a run of 4 pixels of one row. Background + tile layer are a GATHER through a table
//               resolved once per frame: rowcell[tile row][screen column] = atlas address of the top-most tile of that
//               tile row under that column (texture + source column already folded in), so that a pixel costs one
//               16-byte table read per 4 pixels, one add (the source row) and ONE texel fetch; an opaque texel decides
//               the pixel, a transparent / translucent one (or an ambiguous table entry) takes the ordered slow path.
//   post pass   the same warp then draws the post blits that touch its band, blit by blit in submission order
//               (lanes = an 8x4 patch of the blit's destination rectangle), onto the RGBA words (two channels per
//               multiply in the integer SRC-over).
//   store       the band is packed RGBA -> RGB in place (byte permutes) and leaves the SM as one 1 536-byte TMA bulk
//               store (cp.async.bulk.global.shared::cta); cached base images (G::STATIC_VIEW) come in the same way,
//               as one 2 048-byte TMA bulk load per band (cp.async.bulk.shared::cta.global + mbarrier).
//
// The tile layer exploits that render_texture() is separable: a tile's destination columns only
// depend on its x index and its rows only on its y index, so a frame needs <= 32 column and <= 32
// row descriptors instead of up to 27x27 blit records; per screen column / row the (at most two) covering
// tile columns / rows and their source texel indices are tabulated once per frame (ColDesc / RowDesc).
#pragma once
#include "pg2_common.cuh"

namespace pg2 {

constexpr int MAX_WIN = 32;        // tile window extent per axis (maze: 27)
constexpr int MAX_PRE = 2;
#ifndef PG2_RENDER_THREADS
#define PG2_RENDER_THREADS 128
#endif
constexpr int RENDER_THREADS = PG2_RENDER_THREADS;
// Threads of a render CTA as a compile-time constant (every render kernel is launched with RENDER_THREADS; the host-sim
// harness runs one "thread"): strided loops get constant trip counts instead of a division by blockDim.x.
constexpr int CTA_THREADS = WARP_LANES == 32 ? RENDER_THREADS : 1;
constexpr uint8_t NO_TILE = 0xff;
#ifndef PG2_BAND_ROWS
#define PG2_BAND_ROWS 8
#endif
constexpr int BAND_ROWS = PG2_BAND_ROWS, NUM_BANDS = OBS_H / BAND_ROWS, BAND_BYTES = BAND_ROWS * OBS_W * 3, BAND_PX = BAND_ROWS * OBS_W;

// std::sort permutation table (SURVEY Q5). System_Sprite_Render::update sorts (z, entity) pairs
// by z with std::sort (common_systems.cpp:36-38); every sprite of a game has the same z, so the
// comparator is always false and the resulting permutation depends on n only. It is computed on
// the host with the real std::sort (sort_perm.h) and uploaded: sorted[k] = input[perm[n][k]].
constexpr int SORT_MAXN = 256;   // chaser extreme draws 198 sprites (f.live holds 256 ids)
#ifdef PG2_HOSTSIM
static const uint8_t* g_sort_perm = nullptr;
#else
__device__ const uint8_t* g_sort_perm;
#endif
PG2_DEV int sort_perm(int n, int k) { return (n <= 16 || n > SORT_MAXN) ? k : g_sort_perm[n * SORT_MAXN + k]; }

struct BlitRot {
    double s, c;       // sin/cos of the blit angle (deterministic, see sincos_deg)
    int16_t x_lo, x_hi, y_lo, y_hi;   // pixel bounds (inclusive) of the rotated rect's axis-aligned bounding box (rotated_bounds)
};

// Per-pixel form of a blit (what the frame keeps): coverage test = two unsigned compares, sampling = one
// multiply-add + shift per axis (a horizontal flip is folded into hx / incx, which wrap modulo 2^32 to the
// exact non-negative value), texel address = base + sy * tex_w + sx.
// A rotated blit is mapped about the centre of its WHOLE integer rect, which can be of any size: it keeps the rect in
// 32-bit fields instead (rw / rh, and the origin in hx / hy, whose sample phase is always inc / 2: rotated blits are
// never flipped or clipped).
struct alignas(16) FastBlit {
    union {
        struct { int16_t x0, y0; uint16_t w, h; };   // un-rotated: integer destination rect (SDL truncates the float rect)
        struct { uint32_t rw, rh; };                 // rotated: width and height of the rect
    };
    uint32_t hx, incx;                          // un-rotated: sx = (hx + i * incx) >> 16; rotated: hx = x0 (int32)
    uint32_t hy, incy, base;                    // (the same for y); base = tex_offset + s0y * tex_w + s0x
    uint16_t tex_w; uint8_t flags, alpha_mod;   // flags: 1 blend, 2 rotated, 4 invisible
};
static_assert(sizeof(FastBlit) == 32, "FastBlit is two 16-byte words");

constexpr int MAX_TILE_TEX = 32;

// Tile layer + background under one screen column: clo = first covering tile column of the window; per texture
// shape class (textures of one class share width and height) and candidate j (tile column clo + j) a validity bit
// and the source texel x. vc masks are in "candidate index" form (candidate q = jr * 2 + jc): 0b0101 for jc = 0,
// 0b1010 for jc = 1, so that (cw & rw) >> (8 + 4 * cls) is the set of candidates whose class-cls axes cover the pixel.
// Stored as three word arrays indexed by col_slot(X), so that the 16 lanes of a row (lane l owns columns 4l .. 4l+3)
// read consecutive words: no bank conflicts.
struct ColDesc {
    uint32_t cw;       // clo | vc[0] << 8 | vc[1] << 12
    uint32_t csx;      // sx[cls][j] in byte cls * 2 + j
    int32_t pre_sx;    // background: source x under this column, -1: not covered
};
PG2_DEV int col_slot(int X) { return (X >> 2) | (X & 3) << 4; }
// Window cell: atlas offset of the tile's texture | blend << 28 | shape class << 29 | 1 << 31; 0 = no tile.
constexpr uint32_t CELL_OFFSET_MASK = 0x0fffffffu, CELL_PRESENT = 0x80000000u;
// Same for one screen row, plus the tile presence bitmaps of the two candidate tile rows (bit = tile column).
struct alignas(16) RowDesc {
    uint32_t rw;       // rlo | vr[0] << 8 | vr[1] << 12 | rlo * MAX_WIN << 16   (vr: 0b0011 for jr = 0, 0b1100 for jr = 1)
    int32_t pre_row;   // background: tex_offset + sy * tex_w under this row, -1: not covered
    uint32_t syw[2];   // [cls]: (sy * tex_w) of candidate row 0 | candidate row 1 << 16
};
// Candidate slot of a screen column / row, written by the make_axis job of the tile column / row that covers it
// (FrameT::cslot / rslot, [(cls * 2 + (tile index & 1)) * 64 + pixel]: the at most two tile columns that cover a pixel are
// neighbours, so they differ in parity and never share a slot): valid | tile index << 16 | source sample.
constexpr uint32_t SLOT_VALID = 0x80000000u;
// pre_row / pre_sx of a screen row / column the background does not cover, as the base pass sees them (see raster_band_fast)
constexpr uint32_t BG_HOLE = 0x40000000u;

// What the base pass reads per screen row (one 16-byte word): the (at most two) tile rows that cover it, top-most first.
// ra / rb index rows of FrameT::rowcell (WINR = the always-empty row: "none"); cov bit 2 * j + cls: tile row j (0 = a,
// 1 = b) covers this screen row for tiles of shape class cls; syw = sy * tex_w per class (class 0 | class 1 << 16).
struct alignas(16) RowFast {
    uint32_t sywa, sywb;
    int32_t pre_row;   // background: tex_offset + sy * tex_w under this row, -1: not covered
    uint32_t meta;     // ra | rb << 8 | cov << 16
};
// rowcell entry: atlas offset of the tile texture + source x | ambiguous << 28 | shape class << 29 | present << 31.
// Ambiguous: two tiles of different shape classes share the entry's tile row under this column, so which one is on
// top depends on the screen row (the slow path decides).
constexpr uint32_t RC_ADDR_MASK = 0x0fffffffu, RC_AMBIGUOUS = 1u << 28, RC_PRESENT = 0x80000000u;

// Frame description of ONE environment, in shared memory. MAXP = capacity of the post-blit list (per game),
// ROT = whether the game ever rotates a blit (bossfight, caveflyer, jumper HUD).
template <int MAXP, bool ROT, int NCLS, int WINR_, int UNROLL_ = 1>
struct FrameT {
    static constexpr int MAX_POST = MAXP, NROT = ROT ? MAXP : 1, WINR = WINR_;
    static constexpr int BLIT_UNROLL = UNROLL_;   // 8x4 patches of an un-rotated post blit whose texel fetches are in flight together
    static constexpr bool ROTATES = ROT;
    alignas(128) uint32_t band_px[RENDER_THREADS / 32][BAND_PX];     // per warp: the band it is drawing, RGBA words (packed to RGB in place before the store)
    alignas(16) uint32_t rowcell[(WINR_ + 1) * OBS_W];                // [tile row of the window][screen column], + the always-empty row
    RowFast rowf[OBS_H];
    alignas(8) uint64_t mbar[RENDER_THREADS / 32];                    // per warp: mbarrier of its TMA bulk loads
    uint32_t mbar_phase[RENDER_THREADS / 32];
    // ---- the view: everything the rasteriser needs of background + tile layer
    alignas(16) uint32_t col_cw[OBS_W];         // ColDesc fields, indexed by col_slot(X)
    uint32_t col_csx[OBS_W];
    int32_t col_pre[OBS_W];
    RowDesc rowd[OBS_H];
    uint32_t cell[(WINR_ + 1) * MAX_WIN];       // window cells (+1 row: branch-free reads)
    FastBlit fpre[MAX_PRE];
    int npre;
    int wide;                                   // the frame needs the general ordered path for every pixel (never observed)
    int pre_blend;                              // background texture carries alpha
    // ---- per frame
    float view_w, view_h;                       // camera_size of this frame: 64x64, or the window size of a human-mode frame
    int human;                                  // human-mode frame (render_game(false)): general ordered path, any size
    int reuse;                                  // the base image comes from the env's cache: the view is not built
    int overflow;                               // the tile window has more rows than WINR (a sizing error: reported as fault bit 8)
    FastBlit fpost[MAXP];
    BlitRot post_rot[NROT];
    Blit pre[MAX_PRE];
    int npost;
    // tile layer: window origin (tile coordinates, y in render space), extents, descriptors per texture shape class
    int tx0, ty0, ncol, nrow, nclass;
    Axis col[NCLS][MAX_WIN];                    // (read by the general ordered path only)
    Axis row[NCLS][MAX_WIN];
    alignas(16) uint32_t cslot[NCLS * 2 * OBS_W];   // candidate slots of the screen columns / rows, see SLOT_VALID
    uint32_t rslot[NCLS * 2 * OBS_W];
    uint16_t bandmask[MAXP];                    // post blit k touches band b <=> bit b
    uint8_t live[256];                          // live_list(): ids of the live sprites in set order
    int wcount[2][RENDER_THREADS / 32];         // emit_post_blits: visible blits per warp (double-buffered by round)
    int next_band;                              // dynamic hand-out of the row bands to warps
    int class_w[2];                             // texture width of the tile shape classes
    uint32_t tileword[MAX_TILE_TEX];            // per CTA (filled once): window cell word of every tile texture id
};

// Deterministic sin/cos in degrees, mirrored operation by operation from oracle/raster.c
// (pg2o_sincos_deg): IEEE double add/mul only, fixed order, no FMA.
PG2_DEV_CALL void sincos_deg(double deg, double* s, double* c) {
    double r = fmod(deg, 360.0);
    if (r < 0.0) r = __dadd_rn(r, 360.0);
    int q = (int)__ddiv_rn(__dadd_rn(r, 45.0), 90.0);
    double t = __dsub_rn(r, __dmul_rn((double)q, 90.0));
    double x = __dmul_rn(t, 0.017453292519943295);
    double x2 = __dmul_rn(x, x);
    double ps = -1.0 / 355687428096000.0;
    ps = __dadd_rn(__dmul_rn(ps, x2), 1.0 / 1307674368000.0);
    ps = __dsub_rn(__dmul_rn(ps, x2), 1.0 / 6227020800.0);
    ps = __dadd_rn(__dmul_rn(ps, x2), 1.0 / 39916800.0);
    ps = __dsub_rn(__dmul_rn(ps, x2), 1.0 / 362880.0);
    ps = __dadd_rn(__dmul_rn(ps, x2), 1.0 / 5040.0);
    ps = __dsub_rn(__dmul_rn(ps, x2), 1.0 / 120.0);
    ps = __dsub_rn(__dmul_rn(ps, x2), 1.0 / 6.0);
    double s0 = __dadd_rn(x, __dmul_rn(x, __dmul_rn(x2, ps)));
    double pc = 1.0 / 20922789888000.0;
    pc = __dsub_rn(__dmul_rn(pc, x2), 1.0 / 87178291200.0);
    pc = __dadd_rn(__dmul_rn(pc, x2), 1.0 / 479001600.0);
    pc = __dsub_rn(__dmul_rn(pc, x2), 1.0 / 3628800.0);
    pc = __dadd_rn(__dmul_rn(pc, x2), 1.0 / 40320.0);
    pc = __dsub_rn(__dmul_rn(pc, x2), 1.0 / 720.0);
    pc = __dadd_rn(__dmul_rn(pc, x2), 1.0 / 24.0);
    pc = __dsub_rn(__dmul_rn(pc, x2), 0.5);
    double c0 = __dadd_rn(1.0, __dmul_rn(x2, pc));
    switch (q & 3) {
    case 0: *s = s0;  *c = c0;  break;
    case 1: *s = c0;  *c = -s0; break;
    case 2: *s = -s0; *c = -c0; break;
    default: *s = -c0; *c = s0; break;
    }
}

// ---- blit construction helpers (called by the per-game frame builders) --------------------

// Work item k of a frame builder runs on the first lane of warp k (any thread when simulated).
PG2_DEV bool is_role(int k) { return (int)threadIdx.x == (k * 32) % CTA_THREADS; }

// gr.camera_position / gr.camera_scale / gr.camera_size (renderer.h:18-20). The size is 64x64 for observations and the
// window size for the human-mode frame of cenv_render (render_game(false), coinrun.cpp:451-455).
struct Camera { float x, y, scale, w = 64.0f, h = 64.0f; };

// Renderer::render_texture (renderer.cpp:5-82)
PG2_DEV Blit make_blit(const TexInfo* tex, int tex_id, float px, float py, const Camera& cam,
                                          float scale, float alpha = 1.0f, bool flip_h = false) {
    TexInfo t = tex[tex_id];
    Blit b;
    make_axis_xy(px, py, cam.x, cam.y, cam.scale, cam.w, cam.h, t.w, t.h, scale, flip_h, &b.ax, &b.ay);
    if (!b.ay.visible) b.ax.visible = 0;
    b.tex_offset = t.offset; b.tex_w = t.w; b.blend = (uint8_t)t.blend;
    // `SDL_SetTextureAlphaMod(tex, 255 * alpha)`: float -> Uint8 truncation (renderer.cpp:57)
    b.alpha_mod = (alpha != 1.0f) ? (uint8_t)f2i(__fmul_rn(255.0f, alpha)) : (uint8_t)255;
    b.flip_h = flip_h; b.rotated = 0;
    return b;
}

// Renderer::render_texture_rotated (renderer.cpp:84-101): whole texture, no culling / cropping,
// angle = rotation * 180.0f / M_PI evaluated in double (SURVEY Q12).
PG2_DEV Blit make_blit_rotated(const TexInfo* tex, int tex_id, float px, float py, const Camera& cam,
                                                  float rotation, float scale, float alpha, BlitRot* rot) {
    TexInfo t = tex[tex_id];
    Blit b;
    float dx = __fadd_rn(__fmul_rn(__fsub_rn(px, cam.x), cam.scale), __fmul_rn(cam.w, 0.5f));
    float dy = __fadd_rn(__fmul_rn(__fsub_rn(py, cam.y), cam.scale), __fmul_rn(cam.h, 0.5f));
    float dw = __fmul_rn(__fmul_rn((float)t.w, scale), cam.scale);
    float dh = __fmul_rn(__fmul_rn((float)t.h, scale), cam.scale);
    b.ax = make_axis_direct(dx, dw, t.w);
    b.ay = make_axis_direct(dy, dh, t.h);
    if (!b.ay.visible) b.ax.visible = 0;
    b.tex_offset = t.offset; b.tex_w = t.w; b.blend = (uint8_t)t.blend;
    b.alpha_mod = (alpha != 1.0f) ? (uint8_t)f2i(__fmul_rn(255.0f, alpha)) : (uint8_t)255;
    b.flip_h = 0;
    double angle = __ddiv_rn((double)__fmul_rn(rotation, 180.0f), 3.14159265358979323846);
    b.rotated = (angle != 0.0) ? 1 : 0;
    rot->s = 0.0; rot->c = 1.0;
    if (b.rotated) sincos_deg(angle, &rot->s, &rot->c);
    return b;
}

// Blit with an explicit float destination rect and angle in degrees (jumper HUD, jumper.cpp:487-508)
PG2_DEV Blit make_blit_rect(const TexInfo* tex, int tex_id, float dx, float dy, float dw, float dh,
                                               double angle_deg, BlitRot* rot) {
    TexInfo t = tex[tex_id];
    Blit b;
    b.ax = make_axis_direct(dx, dw, t.w);
    b.ay = make_axis_direct(dy, dh, t.h);
    if (!b.ay.visible) b.ax.visible = 0;
    b.tex_offset = t.offset; b.tex_w = t.w; b.blend = (uint8_t)t.blend;
    b.alpha_mod = 255; b.flip_h = 0;
    b.rotated = (angle_deg != 0.0) ? 1 : 0;
    rot->s = 0.0; rot->c = 1.0;
    if (b.rotated) sincos_deg(angle_deg, &rot->s, &rot->c);
    return b;
}

// Wait until every bulk store issued by this thread has finished READING shared memory (see frame_store).
PG2_DEV void frame_store_wait() {
#ifndef PG2_HOSTSIM
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
#endif
}

// vw x vh: the target (64 x 64, or the window of a human-mode frame, at most 32767 pixels per side). An un-rotated rect
// outside the 16-bit fields (never one of a game's observation frames) is clipped to the target first, the skipped
// destination pixels folded into hx / hy (the samples wrap modulo 2^32 exactly like the unclipped ones), so that a rect
// of any size draws what the spec draws. A rotated rect is kept whole in 32-bit fields (see FastBlit).
PG2_DEV FastBlit make_fast(const Blit& b, int vw, int vh) {
    FastBlit fb;
    bool off = false;
    fb.incx = b.flip_h ? 0u - b.ax.inc : b.ax.inc;
    fb.incy = b.ay.inc;
    if (b.rotated) {
        fb.rw = (uint32_t)max(0, b.ax.dlen); fb.rh = (uint32_t)max(0, b.ay.dlen);
        fb.hx = (uint32_t)b.ax.d0; fb.hy = (uint32_t)b.ay.d0;
    } else {
        off = b.ax.d0 < -32768 || b.ax.d0 > 32767 || b.ay.d0 < -32768 || b.ay.d0 > 32767 || b.ax.dlen > 65535 || b.ay.dlen > 65535;
        fb.x0 = (int16_t)b.ax.d0; fb.y0 = (int16_t)b.ay.d0;
        fb.w = (uint16_t)max(0, b.ax.dlen); fb.h = (uint16_t)max(0, b.ay.dlen);
        fb.hx = b.flip_h ? b.ax.inc / 2u + (uint32_t)(b.ax.dlen - 1) * b.ax.inc : b.ax.inc / 2u;
        fb.hy = b.ay.inc / 2u;
    }
    if (__builtin_expect(off && b.ax.visible, 0)) {
        // skip k = -d0 pixels of a rect that starts left of / above the target, keep at most what reaches its far edge
        const uint32_t kx = b.ax.d0 < 0 ? 0u - (uint32_t)b.ax.d0 : 0u, ky = b.ay.d0 < 0 ? 0u - (uint32_t)b.ay.d0 : 0u;
        const int x0 = b.ax.d0 < 0 ? 0 : b.ax.d0, y0 = b.ay.d0 < 0 ? 0 : b.ay.d0;
        const int w = kx >= (uint32_t)b.ax.dlen || x0 >= vw ? 0 : min(b.ax.dlen - (int)kx, vw - x0);
        const int h = ky >= (uint32_t)b.ay.dlen || y0 >= vh ? 0 : min(b.ay.dlen - (int)ky, vh - y0);
        off = w == 0 || h == 0;
        fb.x0 = (int16_t)x0; fb.y0 = (int16_t)y0; fb.w = (uint16_t)w; fb.h = (uint16_t)h;
        fb.hx = b.flip_h ? fb.hx - kx * b.ax.inc : fb.hx + kx * b.ax.inc;
        fb.hy += ky * b.ay.inc;
    }
    fb.base = b.tex_offset + (uint32_t)b.ay.s0 * b.tex_w + (uint32_t)b.ax.s0;
    fb.tex_w = b.tex_w;
    fb.alpha_mod = b.alpha_mod;
    fb.flags = (uint8_t)((b.blend ? 1 : 0) | (b.rotated ? 2 : 0) | ((b.ax.visible && !off) ? 0 : 4));
    return fb;
}

// Pixel bounds of the axis-aligned bounding box of a rotated destination rect. A pixel centre (X + 0.5, Y + 0.5) passes the
// inverse-mapping test of rotated_texel_coords only if |u| <= hw and |v| <= hh, hence |X + 0.5 - cx| <= hw |c| + hh |s| (and
// the same with s, c swapped in y), cx = x0 + hw the real centre. The bounds are rounded OUTWARDS after widening by 1e-3 for
// the rounding of the test's own arithmetic: a bound only has to be conservative, it never changes which pixels are drawn
// (bullets a few pixels long got 9-11 px boxes from the integer centre +- (ceil + 2) of round 1: three times the patches).
PG2_DEV void rotated_bounds(const FastBlit& fb, BlitRot* rot) {
    const double hw = 0.5 * (double)fb.rw, hh = 0.5 * (double)fb.rh, ac = fabs(rot->c), as = fabs(rot->s);
    const double ex = hw * ac + hh * as + 1e-3, ey = hw * as + hh * ac + 1e-3;
    const double cx = (double)(int32_t)fb.hx + hw - 0.5, cy = (double)(int32_t)fb.hy + hh - 0.5;   // pixel index X = centre coordinate - 0.5
    const double lo_x = floor(cx - ex), hi_x = ceil(cx + ex), lo_y = floor(cy - ey), hi_y = ceil(cy + ey);
    rot->x_lo = (int16_t)fmax(lo_x, -32768.0); rot->x_hi = (int16_t)fmin(hi_x, 32767.0);
    rot->y_lo = (int16_t)fmax(lo_y, -32768.0); rot->y_hi = (int16_t)fmin(hi_y, 32767.0);
}

// Bands (8 rows each) a blit can touch.
PG2_DEV uint32_t blit_bands(const FastBlit& fb, const BlitRot& rot) {
    int y0 = fb.y0, y1 = fb.y0 + fb.h - 1;
    if (fb.flags & 2u) { y0 = rot.y_lo; y1 = rot.y_hi; }
    if (y1 < 0 || y0 >= OBS_H) return 0u;
    int b0 = max(y0, 0) / BAND_ROWS, b1 = min(y1, OBS_H - 1) / BAND_ROWS;
    return ((2u << b1) - 1u) & ~((1u << b0) - 1u);
}

// What a game's frame builder asks for per post-blit candidate. The expensive part (make_blit and friends) is run by
// emit_post_blits for all lanes of a warp TOGETHER, whatever kind of sprite each lane describes.
struct BlitReq {
    int mode;            // 0: nothing to draw, 1: render_texture, 2: render_texture_rotated, 3: explicit rect + angle
    int tex_id;
    float x, y, w, h;    // mode 1/2: world position in pixels (w, h unused); mode 3: float destination rect
    float scale, alpha, rotation;
    double angle_deg;
    bool flip;
    Camera cam;
    PG2_DEV void plain(int t, float px, float py, const Camera& c, float sc, float al = 1.0f, bool fl = false) {
        mode = 1; tex_id = t; x = px; y = py; cam = c; scale = sc; alpha = al; flip = fl;
    }
    PG2_DEV void rotated(int t, float px, float py, const Camera& c, float rot, float sc, float al, BlitRot*) {
        mode = 2; tex_id = t; x = px; y = py; cam = c; rotation = rot; scale = sc; alpha = al; flip = false;
    }
    PG2_DEV void rect(int t, float dx, float dy, float dw, float dh, double ang, BlitRot*) {
        mode = 3; tex_id = t; x = dx; y = dy; w = dw; h = dh; angle_deg = ang; flip = false;
    }
};

// Ordered, compacting append of post blits by the whole CTA: candidate k (in the reference's
// submission order) is described by thread k % blockDim (make(k, req, rot) fills the request or leaves it empty);
// only visible blits are stored, order preserved through a warp ballot + a prefix over the warps' counts.
// Must be called by every thread of the CTA, once per frame; ONE barrier per 128 candidates.
template <class F, class MakeFn>
PG2_DEV void emit_post_blits(F& f, const TexInfo* tex, int ncand, MakeFn make) {
    const int tid = threadIdx.x, lane = tid % WARP_LANES, warp = tid / WARP_LANES;
    const int nwarps = (CTA_THREADS + WARP_LANES - 1) / WARP_LANES;
    int n = 0, round = 0;
    for (int base = 0; base < ncand; base += CTA_THREADS, round ^= 1) {
        int k = base + tid;
        BlitReq req; BlitRot rot;
        req.mode = 0; rot.s = 0.0; rot.c = 1.0; rot.x_lo = rot.x_hi = rot.y_lo = rot.y_hi = 0;
        if (k < ncand) make(k, req, rot);
        Blit b;
        b.ax.visible = 0;
        if (req.mode == 1) b = make_blit(tex, req.tex_id, req.x, req.y, req.cam, req.scale, req.alpha, req.flip);
        else if (req.mode == 2) b = make_blit_rotated(tex, req.tex_id, req.x, req.y, req.cam, req.rotation, req.scale, req.alpha, &rot);
        else if (req.mode == 3) b = make_blit_rect(tex, req.tex_id, req.x, req.y, req.w, req.h, req.angle_deg, &rot);
        bool vis = req.mode != 0 && b.ax.visible;
        FastBlit fb;
        if (vis) { fb = make_fast(b, (int)f.view_w, (int)f.view_h); vis = !(fb.flags & 4u); }
        uint32_t m = __ballot_sync(0xffffffffu, vis);
        if (lane == 0) f.wcount[round][warp] = __popc(m);
        __syncthreads();
        int before = 0, total = 0;
        for (int w2 = 0; w2 < nwarps; w2++) { int cnt = f.wcount[round][w2]; if (w2 < warp) before += cnt; total += cnt; }
        if (vis) {
            int idx = n + before + __popc(m & ((1u << lane) - 1u));
            if (idx < F::MAX_POST) {
                if (F::ROTATES && (fb.flags & 2u)) rotated_bounds(fb, &rot);
                f.fpost[idx] = fb;
                f.bandmask[idx] = (uint16_t)blit_bands(fb, rot);
                if (F::ROTATES) f.post_rot[idx] = rot;
            }
        }
        n += total;
    }
    if (tid == 0) f.npost = n < F::MAX_POST ? n : F::MAX_POST;
}

// f.live[0 .. count) = the ids id_or_neg(j) >= 0, j < n, in order (the live members of an ECS set whose dead entries
// are skipped by the reference's iteration). Every warp of the CTA computes the whole list redundantly — identical
// values to identical addresses — so no CTA barrier is needed: a warp reads the list after its own __syncwarp().
template <class F, class Fn>
PG2_DEV int live_list(F& f, int n, Fn id_or_neg) {
    const int lane = threadIdx.x % WARP_LANES;
    int cnt = 0;
    for (int base = 0; base < n; base += WARP_LANES) {
        const int j = base + lane;
        const int v = j < n ? id_or_neg(j) : -1;
        const uint32_t m = lane_ballot(v >= 0, lane);
        if (v >= 0 && cnt < 256) f.live[(cnt + __popc(m & ((1u << lane) - 1u))) & 255] = (uint8_t)v;
        cnt += __popc(m);
    }
    __syncwarp();
    return cnt;
}

// Tile window of System_Tilemap::render (tilemap.cpp:294-302): inclusive tile index range.
PG2_DEV void tile_window(const Camera& cam, int* lower_x, int* lower_y, int* upper_x, int* upper_y) {
    float hx = __fdiv_rn(__fmul_rn(cam.w, 0.5f), cam.scale), hy = __fdiv_rn(__fmul_rn(cam.h, 0.5f), cam.scale);
    float ax = __fmul_rn(__fsub_rn(cam.x, hx), PIXELS_TO_UNIT);
    float ay = __fmul_rn(__fsub_rn(cam.y, hy), PIXELS_TO_UNIT);
    float aw = __fdiv_rn(__fmul_rn(cam.w, PIXELS_TO_UNIT), cam.scale), ah = __fdiv_rn(__fmul_rn(cam.h, PIXELS_TO_UNIT), cam.scale);
    *lower_x = f2i(floorf(ax));
    *lower_y = f2i(floorf(ay));
    *upper_x = f2i(ceilf(__fadd_rn(ax, aw)));
    *upper_y = f2i(ceilf(__fadd_rn(ay, ah)));
}

// Games whose camera and tile map are fixed within an episode (G::STATIC_VIEW: maze, chaser, bossfight) keep the BASE
// IMAGE of an env (clear + background + tile layer, 64x64 RGBA words = the band buffers' own format) in HBM: the first
// frame of an episode draws and stores it, the following frames load it band by band (one TMA bulk load each) instead
// of describing and rasterising the tile layer again.
constexpr size_t VIEW_CACHE_BYTES = (size_t)OBS_W * OBS_H * 4;
constexpr int BAND_CACHE_BYTES = BAND_PX * 4;

struct alignas(16) Word16 { uint32_t a, b, c, d; };

// Start of a frame (every thread; followed by a __syncthreads() before the game's frame builder runs). `reuse`: the base
// image comes from the env's cache (G::STATIC_VIEW), so the view is not built.
template <class F>
PG2_DEV void frame_begin(F& f, bool reuse = false) {   // `reuse` is only looked at by thread 0 (which knows the env)
    const int tid = threadIdx.x;
    if (tid == 0) {
        f.npost = 0; f.ncol = 0; f.nrow = 0; f.nclass = 1; f.next_band = 0; f.reuse = reuse ? 1 : 0; f.overflow = 0;
        f.view_w = (float)OBS_W; f.view_h = (float)OBS_H; f.human = 0;
        if (!reuse) { f.npre = 0; f.wide = 0; f.pre_blend = 0; }
    }
    // cslot and rslot are adjacent: one run of 16-byte words
    for (int k = tid; k < (int)(sizeof(f.cslot) + sizeof(f.rslot)) / 16; k += CTA_THREADS) ((Word16*)f.cslot)[k] = Word16{ 0u, 0u, 0u, 0u };
}

// One band of the base image: cache -> band buffer as ONE 2 048-byte TMA bulk load (async proxy, completion on the
// warp's mbarrier), band buffer -> cache as 16-byte words (first frame of an episode only).
template <class F>
PG2_DEV void band_from_cache(F& f, int warp, uint32_t* buf, const uint8_t* __restrict__ cache_band, int lane) {
#ifdef PG2_HOSTSIM
    memcpy(buf, cache_band, BAND_CACHE_BYTES);
    (void)f; (void)warp; (void)lane;
#else
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&f.mbar[warp]);
    const uint32_t phase = f.mbar_phase[warp];
    __syncwarp();   // every lane has read the phase and is done with the buffer (generic proxy)
    if (lane == 0) {
        f.mbar_phase[warp] = phase ^ 1u;
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(buf);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // earlier generic-proxy accesses of the buffer -> async proxy
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "n"(BAND_CACHE_BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(dst), "l"(cache_band), "n"(BAND_CACHE_BYTES), "r"(bar) : "memory");
    }
    uint32_t done = 0;
    while (!done)
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(bar), "r"(phase) : "memory");
#endif
}
PG2_DEV void band_to_cache(const uint32_t* buf, uint8_t* __restrict__ cache_band, int lane) {
    for (int i = lane; i < BAND_CACHE_BYTES / 16; i += WARP_LANES) ((Word16*)cache_band)[i] = ((const Word16*)buf)[i];
}

// Background + tile layer of a frame (the "pre" blit of render_game and System_Tilemap::render, tilemap.cpp:294-320),
// called by every thread of the CTA from the game's frame builder:
//   - the two axes of the background blit (texture bg_tex at world pixel position (bg_x, bg_y), scale bg_scale) and the
//     window's column / row axes per texture shape class (class_tex(cls) = a texture of that class) are independent
//     make_axis jobs: one job per thread, counted down from the CTA's LAST thread (the first warps build post blits
//     meanwhile), all running the same instruction stream;
//   - the window's cells (tile_at(x, y): tile texture id or NO_TILE; x = window column + lx, y = render-space tile row)
//     and the per-row presence bitmaps, one warp per tile row.
// Every tile axis also registers itself, with its source samples, in the candidate slots of the screen columns / rows it
// covers (cslot / rslot, zeroed by frame_begin).
template <class F, class ClassTex, class TileAt>
PG2_DEV void build_tile_layer(F& f, const Camera& cam, const TexInfo* tex, int nclass, int lx, int ly, int ncol, int nrow,
                              ClassTex class_tex, TileAt tile_at, int bg_tex, float bg_x, float bg_y, float bg_scale) {
    const int tid = threadIdx.x, lane = tid % WARP_LANES, warp = tid / WARP_LANES;
    const int nwarps = (CTA_THREADS + WARP_LANES - 1) / WARP_LANES;
    if (f.reuse) return;   // the base image comes from the env's cache: no descriptors, cells or background needed
    if (nrow > F::WINR) { nrow = F::WINR; if (tid == 0) f.overflow = 1; }
    const int per = ncol + nrow, njobs = 2 + nclass * per;
    if (tid == 0) { f.tx0 = lx; f.ty0 = ly; f.ncol = ncol; f.nrow = nrow; f.nclass = nclass; f.npre = 1; }
    // window cells: lanes = tile columns, two tile rows per warp pass when the window is at most 16 columns wide
    // (cells right of the window stay unwritten: nothing valid ever points at them). The tile loads of the first two
    // passes are issued here, so that their latency runs under the axis jobs below.
    const int cpr = ncol <= 16 ? 16 : 32, rpp = 32 / cpr;
    constexpr int CELL_AHEAD = WARP_LANES == 32 ? 2 : 0;
    uint32_t ahead[CELL_AHEAD > 0 ? CELL_AHEAD : 1];
#pragma unroll
    for (int q = 0; q < CELL_AHEAD; q++) {
        const int ry = (warp + q * nwarps) * rpp + lane / cpr, cx = lane % cpr;
        ahead[q] = (ry < nrow && cx < ncol) ? (uint32_t)tile_at(lx + cx, ly + ry) : (uint32_t)NO_TILE;
    }
    for (int job = CTA_THREADS - 1 - tid; job < njobs; job += CTA_THREADS) {
        const bool bg = job < 2;
        const int t = job - 2, cls = (!bg && t >= per) ? 1 : 0, u = bg ? 0 : t - cls * per;
        const bool is_row = bg ? job == 1 : u >= ncol;
        const int idx = is_row ? u - ncol : u;
        const TexInfo ti = tex[bg ? bg_tex : class_tex(cls)];
        const float scale = bg ? bg_scale : __fdiv_rn(UNIT_TO_PIXELS, (float)ti.w);
        const float pos = bg ? (is_row ? bg_y : bg_x) : __fmul_rn((float)((is_row ? ly : lx) + idx), UNIT_TO_PIXELS);
        const Axis a = make_axis(pos, is_row ? cam.y : cam.x, cam.scale, is_row ? cam.h : cam.w, is_row ? ti.h : ti.w, scale, false, is_row);
        if (bg) {
            if (is_row) f.pre[0].ay = a;
            else {   // the x-axis job also fills the rest of the blit (make_blit, alpha 1, no flip)
                f.pre[0].ax = a;
                f.pre[0].tex_offset = ti.offset; f.pre[0].tex_w = ti.w; f.pre[0].blend = (uint8_t)ti.blend;
                f.pre[0].alpha_mod = 255; f.pre[0].flip_h = 0; f.pre[0].rotated = 0;
            }
            continue;
        }
        if (is_row) f.row[cls][idx] = a; else f.col[cls][idx] = a;
        if (f.human) continue;   // window-size frame: drawn by the general ordered path from the axes themselves
        if (a.visible && a.d0 > -65536 && a.d0 < 65536 && a.dlen < 65536) {
            // register in the candidate slot of every screen column / row this tile column / row covers, with the source
            // sample under it (rows: already multiplied by the texture width); a slot that was taken means three tiles
            // cover one pixel: the frame goes the general ordered way
            const int p0 = max(a.d0, 0), p1 = min(a.d0 + a.dlen - 1, OBS_W - 1);
            uint32_t* slot = (is_row ? f.rslot : f.cslot) + (cls * 2 + (idx & 1)) * OBS_W;
            const uint32_t mul = is_row ? (uint32_t)ti.w : 1u, lim = is_row ? 0xffffu : 0xffu;
            uint32_t acc = a.inc / 2u + (uint32_t)(p0 - a.d0) * a.inc;
            bool bad = false;
            for (int pp = p0; pp <= p1; pp++, acc += a.inc) {
                const uint32_t v = ((uint32_t)a.s0 + (acc >> 16)) * mul;
                if (v > lim) bad = true;
                if (atomicExch(&slot[pp], SLOT_VALID | (uint32_t)idx << 16 | (v & 0xffffu)) != 0u) bad = true;
            }
            if (bad) f.wide = 1;
        }
    }
    for (int cls = tid; cls < nclass; cls += CTA_THREADS) f.class_w[cls] = tex[class_tex(cls)].w;
#pragma unroll
    for (int q = 0; q < CELL_AHEAD; q++) {
        const int ry = (warp + q * nwarps) * rpp + lane / cpr, cx = lane % cpr;
        if (ry < nrow) f.cell[ry * MAX_WIN + cx] = ahead[q] != NO_TILE ? f.tileword[ahead[q] & (MAX_TILE_TEX - 1)] : 0u;
    }
    for (int ry0 = (warp + CELL_AHEAD * nwarps) * rpp; ry0 < nrow; ry0 += nwarps * rpp)
        for (int l = lane; l < 32; l += WARP_LANES) {
            const int ry = ry0 + l / cpr, cx = l % cpr;
            if (ry < nrow) {
                const uint32_t tt = cx < ncol ? (uint32_t)tile_at(lx + cx, ly + ry) : (uint32_t)NO_TILE;
                f.cell[ry * MAX_WIN + cx] = tt != NO_TILE ? f.tileword[tt & (MAX_TILE_TEX - 1)] : 0u;
            }
        }
}

// ---- per-pixel evaluation ---------------------------------------------------------------------

// After the game's frame builder (and a __syncthreads()): the per-column / per-row tables of the base pass, from the
// candidate slots the axis jobs filled. Job k < 64: screen column k (ColDesc, background x, rowcell entries of the even
// tile rows); job 64 + k: screen row k (RowDesc, RowFast) and the rowcell entries of column k for the odd tile rows.
template <class G, class F>
PG2_DEV_NOINLINE void frame_finalize(F& f) {
    if (f.reuse) { __syncthreads(); return; }
    constexpr int NCLS = G::TILE_CLASSES;
    const int tid = threadIdx.x;
    const int npre = f.npre, nrow = f.nrow;
    // the fast path handles ONE un-rotated background with alpha_mod 255
    const bool pre_ok = npre == 0 || (npre == 1 && !f.pre[0].rotated && f.pre[0].alpha_mod == 255);
    if (tid == 0) {
        if (!pre_ok) f.wide = 1;
        f.pre_blend = npre >= 1 ? f.pre[npre - 1].blend : 0;
    }
    for (int k = tid; k < npre; k += CTA_THREADS) {
        Blit b = f.pre[k];
        if (!b.ay.visible) b.ax.visible = 0;   // make_blit's rule (the two axes were built by different threads)
        f.fpre[k] = make_fast(b, (int)f.view_w, (int)f.view_h);
    }
    if (f.human) {   // window-size frame: no 64-pixel tables, every pixel goes the general ordered way
        if (tid == 0) f.wide = 1;
        __syncthreads();
        return;
    }
    for (int k = tid; k < 2 * OBS_W; k += CTA_THREADS) {
        const bool is_row = k >= OBS_W;
        const int p = k & (OBS_W - 1);
        // the column's candidates (always needed: both jobs of a column build rowcell entries)
        const uint32_t* cs = f.cslot + p;
        uint32_t cw[NCLS][2];
        int clo = 255, chi = -1;
#pragma unroll
        for (int cls = 0; cls < NCLS; cls++)
#pragma unroll
            for (int par = 0; par < 2; par++) {
                const uint32_t w = G::HAS_TILES ? cs[(cls * 2 + par) * OBS_W] : 0u;
                cw[cls][par] = w;
                if (w) { const int idx = (int)(w >> 16 & 31u); clo = min(clo, idx); chi = max(chi, idx); }
            }
        if (chi - clo > 1) f.wide = 1;
        // candidate j of class cls = the slot of parity (clo + j) & 1
        uint32_t cword = chi >= 0 ? (uint32_t)clo : 0u, csx = 0u;
        uint32_t cj[NCLS][2];
#pragma unroll
        for (int cls = 0; cls < NCLS; cls++)
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const uint32_t w = chi >= 0 ? ((clo + j) & 1 ? cw[cls][1] : cw[cls][0]) : 0u;
                cj[cls][j] = w;
                if (w) { cword |= (j ? 0xau : 0x5u) << (8 + 4 * cls); csx |= (w & 255u) << (8 * (cls * 2 + j)); }
            }
        if (!is_row) {
            int32_t pv = -1;
            if (npre >= 1 && pre_ok) {
                const Blit& b = f.pre[0];
                if (b.ax.visible && b.ay.visible && (unsigned)(p - b.ax.d0) < (unsigned)b.ax.dlen) pv = axis_sample(b.ax, p, b.flip_h != 0);
            }
            const int slot = col_slot(p);
            f.col_cw[slot] = cword; f.col_csx[slot] = csx; f.col_pre[slot] = pv;
        } else {
            const uint32_t* rs = f.rslot + p;
            uint32_t rwv[NCLS][2];
            int lo = 255, hi = -1;
#pragma unroll
            for (int cls = 0; cls < NCLS; cls++)
#pragma unroll
                for (int par = 0; par < 2; par++) {
                    const uint32_t w = G::HAS_TILES ? rs[(cls * 2 + par) * OBS_W] : 0u;
                    rwv[cls][par] = w;
                    if (w) { const int idx = (int)(w >> 16 & 31u); lo = min(lo, idx); hi = max(hi, idx); }
                }
            if (hi - lo > 1) f.wide = 1;
            uint32_t word = hi >= 0 ? (uint32_t)lo : 0u, smp[2] = { 0u, 0u };
#pragma unroll
            for (int cls = 0; cls < NCLS; cls++)
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    const uint32_t w = hi >= 0 ? ((lo + j) & 1 ? rwv[cls][1] : rwv[cls][0]) : 0u;
                    if (w) { word |= (j ? 0xcu : 0x3u) << (8 + 4 * cls); smp[cls] |= (w & 0xffffu) << (16 * j); }
                }
            int32_t pv = -1;
            if (npre >= 1 && pre_ok) {
                const Blit& b = f.pre[0];
                if (b.ax.visible && b.ay.visible && (unsigned)(p - b.ay.d0) < (unsigned)b.ay.dlen)
                    pv = (int32_t)(b.tex_offset + (uint32_t)axis_sample(b.ay, p, false) * b.tex_w);
            }
            RowDesc rd;
            rd.rw = word | ((hi >= 0 ? (uint32_t)lo : 0u) * MAX_WIN) << 16; rd.pre_row = pv; rd.syw[0] = smp[0]; rd.syw[1] = smp[1];
            f.rowd[p] = rd;
            // the base pass's view of the row: tile row a = the top-most covering one (candidate ja), b = the one below
            RowFast rf;
            const uint32_t ja = lo < hi ? 1u : 0u;
            const uint32_t v0 = word >> 8 & 15u, v1 = word >> 12 & 15u;            // class 0 / 1: 0x3 = candidate row 0, 0xc = row 1
            const uint32_t cova = (v0 >> (2u * ja) & 1u) | (v1 >> (2u * ja) & 1u) << 1;
            const uint32_t covb = ja ? ((v0 & 1u) | (v1 & 1u) << 1) : 0u;
            rf.sywa = (smp[0] >> (16u * ja) & 0xffffu) | (smp[1] >> (16u * ja) & 0xffffu) << 16;
            rf.sywb = ja ? ((smp[0] & 0xffffu) | (smp[1] & 0xffffu) << 16) : 0u;
            rf.pre_row = pv < 0 ? (int32_t)BG_HOLE : pv;
            const uint32_t ra = hi >= 0 ? (uint32_t)lo + ja : (uint32_t)F::WINR, rb = ja ? (uint32_t)lo : (uint32_t)F::WINR;
            rf.meta = ra | rb << 8 | (cova | covb << 2) << 16;
            f.rowf[p] = rf;
        }
        // rowcell[tile row][column p]: the top-most tile of the tile row under this screen column (painter's order within a
        // tile row = ascending tile column), texture offset + source x folded in; even tile rows by the column job, odd
        // ones by the row job of the same index
        if (G::HAS_TILES) {
            const bool two = clo < chi;
            for (int r = is_row ? 1 : 0; r < nrow; r += 2) {
                uint32_t e = 0u;
                if (chi >= 0) {
                    const uint32_t w0 = f.cell[r * MAX_WIN + clo], w1 = two ? f.cell[r * MAX_WIN + clo + 1] : 0u;
                    const uint32_t c0 = NCLS > 1 ? w0 >> 29 & 1u : 0u, c1 = NCLS > 1 ? w1 >> 29 & 1u : 0u;
                    const uint32_t s0 = NCLS > 1 && c0 ? cj[NCLS - 1][0] : cj[0][0], s1 = NCLS > 1 && c1 ? cj[NCLS - 1][1] : cj[0][1];
                    const bool ok0 = w0 != 0u && s0 != 0u, ok1 = w1 != 0u && s1 != 0u;
                    if (ok1) {
                        e = (w1 & ~(1u << 28)) + (s1 & 255u);
                        if (NCLS > 1 && ok0 && c0 != c1) e |= RC_AMBIGUOUS;
                    } else if (ok0) {
                        e = (w0 & ~(1u << 28)) + (s0 & 255u);
                    }
                }
                f.rowcell[r * OBS_W + p] = e;
            }
        }
    }
    __syncthreads();
}

// Rotated blit: inverse-map the pixel centre into the un-rotated destination rect (oracle/raster.c step 4).
// (Measured: a real call here costs bossfight / caveflyer ~10 % of the render.)
PG2_DEV bool rotated_texel_coords(int x0, int y0, int w, int h, double rs, double rc, int X, int Y, uint32_t* oi, uint32_t* oj) {
    double hw = __dmul_rn((double)w, 0.5), hh = __dmul_rn((double)h, 0.5);
    double cx = __dadd_rn((double)x0, hw), cy = __dadd_rn((double)y0, hh);
    double px = __dsub_rn(__dadd_rn((double)X, 0.5), cx);
    double py = __dsub_rn(__dadd_rn((double)Y, 0.5), cy);
    double u = __dadd_rn(__dmul_rn(px, rc), __dmul_rn(py, rs));
    double v = __dsub_rn(__dmul_rn(py, rc), __dmul_rn(px, rs));
    double fu = floor(__dadd_rn(u, hw)), fv = floor(__dadd_rn(v, hh));
    if (fu < 0.0 || fv < 0.0 || fu >= (double)w || fv >= (double)h) return false;
    *oi = (uint32_t)(int)fu; *oj = (uint32_t)(int)fv;
    return true;
}

// Texel of a blit under pixel (X, Y); false when the pixel is not covered.
template <bool ROT>
PG2_DEV bool fast_texel(const FastBlit& fb, const BlitRot* rot, const uint32_t* __restrict__ atlas, int X, int Y, uint32_t* texel) {
    uint32_t i, j, hx = fb.hx, hy = fb.hy;
    if (ROT && (fb.flags & 2u)) {
        if (!rotated_texel_coords((int32_t)fb.hx, (int32_t)fb.hy, (int)fb.rw, (int)fb.rh, rot->s, rot->c, X, Y, &i, &j)) return false;
        hx = fb.incx / 2u; hy = fb.incy / 2u;
    } else {
        i = (uint32_t)(X - fb.x0); j = (uint32_t)(Y - fb.y0);
        if (i >= fb.w || j >= fb.h) return false;
    }
    uint32_t sx = (hx + i * fb.incx) >> 16, sy = (hy + j * fb.incy) >> 16;
    *texel = __ldg(atlas + fb.base + sy * fb.tex_w + sx);
    return true;
}

// Effective alpha of a texel of a layer: A * alpha_mod / 255. Opaque-copy (RGB) textures are stored with A = 255 in
// the atlas (assets.cpp), and SRC-over with alpha 255 IS the copy, so the blend flag never needs to be consulted.
PG2_DEV uint32_t layer_alpha(uint32_t texel, uint32_t /*blend*/, uint32_t alpha_mod) {
    uint32_t ta = texel >> 24;
    return alpha_mod != 255u ? (ta * alpha_mod) / 255u : ta;
}

// SRC-over of one texel onto a packed 0x00BBGGRR colour; effective alpha 255 replaces and 0 is the identity
// (both exact in blend_texel's integer arithmetic), anything else takes the full per-channel path.
PG2_DEV uint32_t blend_packed(uint32_t color, uint32_t texel, uint32_t blend, uint32_t alpha_mod) {
    uint32_t a = layer_alpha(texel, blend, alpha_mod);
    if (a == 255u) return texel;
    if (a == 0u) return color;
    uint32_t r = color & 255u, g = (color >> 8) & 255u, b = (color >> 16) & 255u;
    blend_texel(r, g, b, texel, blend, alpha_mod);
    return r | g << 8 | b << 16;
}

// Tile candidates of a pixel as a 4-bit set (candidate q = jr * 2 + jc <=> tile (rlo + jr, clo + jc)): a tile is
// there and the axes of its shape class cover the pixel. Painter's order = ascending q. (Slow path only.)
template <int NCLASS, class F>
PG2_DEV uint32_t tile_candidates(const F& f, const RowDesc& rd, uint32_t cw) {
    const uint32_t v = cw & rd.rw, base = (rd.rw >> 16) + (cw & 31u);
    uint32_t p = 0u;
#pragma unroll
    for (uint32_t q = 0; q < 4u; q++) {
        const uint32_t w = f.cell[base + (q >> 1) * MAX_WIN + (q & 1u)];
        const uint32_t cls = NCLASS > 1 ? w >> 29 & 1u : 0u;
        if (w != 0u && (v >> (8u + 4u * cls) >> q & 1u)) p |= 1u << q;
    }
    return p;
}

template <class F>
PG2_DEV ColDesc load_col(const F& f, int X) {
    const int slot = col_slot(X);
    ColDesc cd;
    cd.cw = f.col_cw[slot]; cd.csx = f.col_csx[slot]; cd.pre_sx = f.col_pre[slot];
    return cd;
}

// Atlas index of tile candidate q under a pixel. q = 2 jr + jc, so the cell (rlo + jr, clo + jc) is at
// rlo * 32 + clo + 30 jr + q; the 8-bit sx / 16-bit sy*w fields are picked with one byte permute each.
template <int NCLASS, class F>
PG2_DEV uint32_t tile_texel_index(const F& f, const RowDesc& rd, const ColDesc& cd, uint32_t q) {
    const uint32_t jr = q >> 1;
    const uint32_t w = f.cell[(rd.rw >> 16) + (cd.cw & 31u) + jr * 30u + q];   // rw >> 16 = rlo * MAX_WIN
    const uint32_t cls = NCLASS > 1 ? (w >> 29) & 1u : 0u;
    const uint32_t sx = byte_perm(cd.csx, 0u, 0x4440u | (cls * 2u + (q & 1u)));
    const uint32_t syw = byte_perm(cls ? rd.syw[1] : rd.syw[0], 0u, 0x4410u + jr * 0x22u);
    return (w & CELL_OFFSET_MASK) + syw + sx;
}

// clear -> pre -> tiles of one pixel in reference (bottom-up) order with full blending: the path of pixels whose
// top-most layer is translucent, and of every pixel of a `wide` frame (more than two tiles cover a column / row,
// or a background the tables do not describe), which walks the covering ranges with the axes themselves.
template <class G, class F>
PG2_DEV_COLD uint32_t shade_base_ordered(const F& f, const uint32_t* __restrict__ atlas, int X, int Y) {
    uint32_t color = 0u, texel;   // SDL_RenderClear(0,0,0,255)
    for (int k = 0; k < f.npre; k++) {
        const FastBlit fb = f.fpre[k];
        BlitRot rot{ 0.0, 1.0, 0, 0, 0, 0 };
        if (!(fb.flags & 4u) && fast_texel<false>(fb, &rot, atlas, X, Y, &texel)) color = blend_packed(color, texel, fb.flags & 1u, fb.alpha_mod);
    }
    if (!f.wide) {
        const RowDesc rd = f.rowd[Y];
        const ColDesc cd = load_col(f, X);
        uint32_t p = tile_candidates<G::TILE_CLASSES>(f, rd, cd.cw);
        for (uint32_t q = 0; q < 4u; q++)
            if (p >> q & 1u) {
                texel = __ldg(atlas + tile_texel_index<G::TILE_CLASSES>(f, rd, cd, q));
                color = blend_packed(color, texel, 1u, 255u);
            }
        return color;
    }
    for (int ry = 0; ry < f.nrow; ry++)       // (never observed: every tile of the window is tested against the pixel)
        for (int cx = 0; cx < f.ncol; cx++) {
            const uint32_t w = f.cell[ry * MAX_WIN + cx];
            if (!w) continue;
            const uint32_t cls = (w >> 29) & 1u;
            const Axis& ax = f.col[cls][cx];
            const Axis& ay = f.row[cls][ry];
            if (!ax.visible || !ay.visible) continue;
            if ((unsigned)(X - ax.d0) >= (unsigned)ax.dlen || (unsigned)(Y - ay.d0) >= (unsigned)ay.dlen) continue;
            int sx = axis_sample(ax, X, false), sy = axis_sample(ay, Y, false);
            texel = __ldg(atlas + (w & CELL_OFFSET_MASK) + (uint32_t)sy * (uint32_t)f.class_w[cls] + (uint32_t)sx);
            color = blend_packed(color, texel, 1u, 255u);
        }
    return color;
}

// A pixel whose top-most tile texel turned out transparent: keep walking its candidates top-down (then the
// background); the first opaque texel decides, a translucent one hands the pixel to shade_base_ordered.
template <class G, class F>
PG2_DEV_COLD uint32_t shade_base_continue(const F& f, const uint32_t* __restrict__ atlas, int X, int Y, uint32_t p) {
    const RowDesc rd = f.rowd[Y];
    const ColDesc cd = load_col(f, X);
    while (p) {
        const uint32_t q = bfind(p);
        p &= ~(1u << q);
        const uint32_t texel = __ldg(atlas + tile_texel_index<G::TILE_CLASSES>(f, rd, cd, q));
        const uint32_t a = texel >> 24;
        if (a == 255u) return texel;
        if (a != 0u) return shade_base_ordered<G>(f, atlas, X, Y);
    }
    if ((rd.pre_row | cd.pre_sx) < 0) return 0u;
    const uint32_t texel = __ldg(atlas + (uint32_t)rd.pre_row + (uint32_t)cd.pre_sx);
    const uint32_t a = texel >> 24;
    if (a == 255u) return texel;
    return a ? shade_base_ordered<G>(f, atlas, X, Y) : 0u;
}

// x / 255 for two 16-bit lanes at once (each lane <= 65 534: exact, no carry between the lanes).
PG2_DEV uint32_t div255x2(uint32_t v) { return ((v + 0x00010001u + ((v >> 8) & 0x00ff00ffu)) >> 8) & 0x00ff00ffu; }
PG2_DEV uint32_t div255(uint32_t v) { return (v + 1u + (v >> 8)) >> 8; }

// SRC-over of one texel with effective alpha a in [1, 254] onto an RGBA word: blend_texel's integer arithmetic
// (premultiply by a, then dst * (255 - a) / 255), red and blue in one multiply.
PG2_DEV uint32_t blend_word(uint32_t dst, uint32_t texel, uint32_t a) {
    const uint32_t ia = 255u - a;
    const uint32_t trb = div255x2((texel & 0x00ff00ffu) * a), tg = div255((texel >> 8 & 255u) * a);
    const uint32_t drb = div255x2((dst & 0x00ff00ffu) * ia), dg = div255((dst >> 8 & 255u) * ia);
    return (trb + drb) | (tg + dg) << 8;
}

// Human-mode frame (cenv_render, render_game(false)): one pixel of a frame of any size — clear, background, every tile of
// the window and every post blit in the reference's order with full blending. The frame was described with the window
// size as camera_size (f.human: no 64-pixel tables are built), f.wide is set.
template <class G, class F>
PG2_DEV uint32_t shade_human_pixel(const F& f, const uint32_t* __restrict__ atlas, int X, int Y) {
    uint32_t color = shade_base_ordered<G>(f, atlas, X, Y);
    for (int k = 0; k < f.npost; k++) {
        const FastBlit fb = f.fpost[k];
        uint32_t texel;
        if (fast_texel<F::ROTATES>(fb, &f.post_rot[F::ROTATES ? k : 0], atlas, X, Y, &texel)) {
            const uint32_t a = (fb.flags & 1u) ? layer_alpha(texel, 1u, fb.alpha_mod) : 255u;
            if (a == 255u) color = texel;
            else if (a != 0u) color = blend_word(color, texel, a);
        }
    }
    return color;
}

// A pixel the base pass could not decide from its table: all tile candidates top-down, then the background.
#ifdef PG2_HOSTSIM
static long g_dbg_slow = 0, g_dbg_quads = 0, g_dbg_quads_slow = 0, g_dbg_rb = 0;   // host-sim statistics (scripts/sim_check.py)
#endif
template <class G, class F>
PG2_DEV_COLD uint32_t shade_base_slow(const F& f, const uint32_t* __restrict__ atlas, int X, int Y) {
#ifdef PG2_HOSTSIM
    g_dbg_slow++;
#endif
    const RowDesc rd = f.rowd[Y];
    const uint32_t p = G::HAS_TILES ? tile_candidates<G::TILE_CLASSES>(f, rd, load_col(f, X).cw) : 0u;
    return shade_base_continue<G>(f, atlas, X, Y, p);
}

// Base pass of one band: clear + background + tile layer of 8 rows as RGBA words in the warp's band buffer.
// A thread owns PG2_BASE_PX consecutive pixels of a row: 16-byte reads of the top tile row's rowcell entries, per pixel
// one add + one select + one texel fetch (independent fetches in flight), 16-byte stores. The second covering tile row is only looked at on the few screen rows that have one.
// A pixel the background does not cover reads the atlas' black texel (index 0 = the clear colour): pre_row / pre_sx of
// an uncovered row / column are BG_HOLE, which no sum of real indices reaches.
#ifndef PG2_BASE_PX
#define PG2_BASE_PX 4   // pixels per thread in the base pass (4 or 8; measured: 4 is 8-10 % faster, fewer live registers)
#endif
template <class G, class F>
PG2_DEV void raster_band_fast(F& f, const uint32_t* __restrict__ atlas, int band, int lane, uint32_t* buf) {
    constexpr int NCLASS = G::TILE_CLASSES, PX = PG2_BASE_PX, LPR = OBS_W / PX, RPP = 32 / LPR;   // lanes per row, rows per pass
    for (int l = lane; l < 32; l += WARP_LANES) {
        const int X0 = (l % LPR) * PX;
        uint32_t pre_sx[PX];
#pragma unroll
        for (int i = 0; i < PX; i++) { const int32_t v = f.col_pre[col_slot(X0 + i)]; pre_sx[i] = v < 0 ? BG_HOLE : (uint32_t)v; }
        for (int it = 0; it < BAND_ROWS / RPP; it++) {
            const int yl = it * RPP + l / LPR, Y = band * BAND_ROWS + yl;
            const RowFast rf = f.rowf[Y];
            uint32_t at[PX], texel[PX], flags = 0u;
#pragma unroll
            for (int i = 0; i < PX; i++) {
                const uint32_t v = (uint32_t)rf.pre_row + pre_sx[i];
                at[i] = v >= BG_HOLE ? 0u : v;
            }
            if (G::HAS_TILES) {
                const uint32_t ra = rf.meta & 255u, rb = rf.meta >> 8 & 255u;
                if (rb != (uint32_t)F::WINR) {   // a second tile row covers this screen row: the lower one first, then a on top
                    uint32_t eb[PX];
#pragma unroll
                    for (int i = 0; i < PX; i += 4) { const Word16 w = *(const Word16*)&f.rowcell[rb * OBS_W + X0 + i]; eb[i] = w.a; eb[i + 1] = w.b; eb[i + 2] = w.c; eb[i + 3] = w.d; }
#pragma unroll
                    for (int i = 0; i < PX; i++) {
                        const uint32_t e = eb[i];
                        if (NCLASS > 1) {
                            const uint32_t cls = e >> 29 & 1u;
                            if ((int32_t)e < 0 && (rf.meta >> (18u + cls) & 1u)) at[i] = (e & RC_ADDR_MASK) + (cls ? rf.sywb >> 16 : rf.sywb & 0xffffu);
                        } else if ((int32_t)e < 0) at[i] = (e & RC_ADDR_MASK) + rf.sywb;
                        flags |= e;
                    }
                }
                uint32_t ea[PX];
#pragma unroll
                for (int i = 0; i < PX; i += 4) { const Word16 w = *(const Word16*)&f.rowcell[ra * OBS_W + X0 + i]; ea[i] = w.a; ea[i + 1] = w.b; ea[i + 2] = w.c; ea[i + 3] = w.d; }
#pragma unroll
                for (int i = 0; i < PX; i++) {
                    const uint32_t e = ea[i];
                    if (NCLASS > 1) {
                        const uint32_t cls = e >> 29 & 1u;
                        if ((int32_t)e < 0 && (rf.meta >> (16u + cls) & 1u)) at[i] = (e & RC_ADDR_MASK) + (cls ? rf.sywa >> 16 : rf.sywa & 0xffffu);
                    } else if ((int32_t)e < 0) at[i] = (e & RC_ADDR_MASK) + rf.sywa;
                    flags |= e;
                }
            }
            uint32_t all = 0xffffffffu;
#pragma unroll
            for (int i = 0; i < PX; i++) { texel[i] = __ldg(atlas + at[i]); all &= texel[i]; }
            // opaque-copy textures carry A = 255 in the atlas: ONE test covers the common case of all-opaque texels
#ifdef PG2_HOSTSIM
            g_dbg_quads++;
            if (G::HAS_TILES && (rf.meta >> 8 & 255u) != (uint32_t)F::WINR) g_dbg_rb++;
            if ((all >> 24) != 255u || (flags & RC_AMBIGUOUS) != 0u) g_dbg_quads_slow++;
#endif
            if ((all >> 24) != 255u || (flags & RC_AMBIGUOUS) != 0u) {
                for (int i = 0; i < PX; i++)
                    if ((flags & RC_AMBIGUOUS) != 0u || (texel[i] >> 24) != 255u) texel[i] = shade_base_slow<G>(f, atlas, X0 + i, Y);
            }
#pragma unroll
            for (int i = 0; i < PX; i += 4) {
                Word16 o; o.a = texel[i]; o.b = texel[i + 1]; o.c = texel[i + 2]; o.d = texel[i + 3];
                *(Word16*)&buf[yl * OBS_W + X0 + i] = o;
            }
        }
    }
}

template <class G, class F>
PG2_DEV void raster_band_base(F& f, const uint32_t* __restrict__ atlas, int band, int lane, uint32_t* buf) {
    if (f.wide != 0) {   // general ordered path for every pixel (never observed)
        for (int it = 0; it < BAND_ROWS / 2; it++)
            for (int l = lane; l < 32; l += WARP_LANES) {
                const int yl = it * 2 + (l >> 4), X0 = (l & 15) * 4;
#pragma unroll
                for (int i = 0; i < 4; i++) buf[yl * OBS_W + X0 + i] = shade_base_ordered<G>(f, atlas, X0 + i, band * BAND_ROWS + yl);
            }
        return;
    }
    raster_band_fast<G>(f, atlas, band, lane, buf);
}

// One post blit onto the rows [Y0, Y0 + 8) (the band buffer): lanes = an 8x4 patch of the destination rectangle.
template <class F>
PG2_DEV void draw_blit_band(F& f, const uint32_t* __restrict__ atlas, int k, int Y0, int lane, uint32_t* buf) {
    const FastBlit fb = f.fpost[k];
    const BlitRot* rot = &f.post_rot[F::ROTATES ? k : 0];
    int x0 = fb.x0, y0 = fb.y0, x1 = fb.x0 + fb.w - 1, y1 = fb.y0 + fb.h - 1;
    if (F::ROTATES && (fb.flags & 2u)) { x0 = rot->x_lo; x1 = rot->x_hi; y0 = rot->y_lo; y1 = rot->y_hi; }   // bounding box of the rotated rect
    x0 = max(x0, 0); x1 = min(x1, OBS_W - 1); y0 = max(y0, Y0); y1 = min(y1, Y0 + BAND_ROWS - 1);
    const uint32_t blend = fb.flags & 1u, alpha_mod = fb.alpha_mod;
    if (!(F::ROTATES && (fb.flags & 2u))) {
        // un-rotated: F::BLIT_UNROLL patches side by side per round, all texel fetches issued before the first blend (games with
        // large sprites: bossfight + 3.5 %; small-sprite games measured 3-10 % slower with it and keep 1)
        for (int yb = y0; yb <= y1; yb += 4)
            for (int xb = x0; xb <= x1; xb += 8 * F::BLIT_UNROLL)
                for (int l = lane; l < 32; l += WARP_LANES) {
                    const int Y = yb + (l >> 3);
                    const uint32_t j = (uint32_t)(Y - fb.y0);
                    const bool row_ok = Y <= y1 && j < fb.h;
                    const uint32_t row = fb.base + ((fb.hy + j * fb.incy) >> 16) * fb.tex_w;
                    uint32_t texel[F::BLIT_UNROLL];
                    bool ok[F::BLIT_UNROLL];
#pragma unroll
                    for (int u = 0; u < F::BLIT_UNROLL; u++) {
                        const int X = xb + 8 * u + (l & 7);
                        const uint32_t i = (uint32_t)(X - fb.x0);
                        ok[u] = row_ok && X <= x1 && i < fb.w;
                        texel[u] = ok[u] ? __ldg(atlas + row + ((fb.hx + i * fb.incx) >> 16)) : 0u;
                    }
#pragma unroll
                    for (int u = 0; u < F::BLIT_UNROLL; u++) {
                        if (!ok[u]) continue;
                        const uint32_t a = blend ? layer_alpha(texel[u], blend, alpha_mod) : 255u;   // an opaque-copy texture ignores the alpha mod
                        uint32_t* px = buf + (Y - Y0) * OBS_W + xb + 8 * u + (l & 7);
                        if (a == 255u) *px = texel[u];
                        else if (a != 0u) *px = blend_word(*px, texel[u], a);
                    }
                }
        __syncwarp();
        return;
    }
    for (int yb = y0; yb <= y1; yb += 4)
        for (int xb = x0; xb <= x1; xb += 8)
            for (int l = lane; l < 32; l += WARP_LANES) {
                const int X = xb + (l & 7), Y = yb + (l >> 3);
                uint32_t texel;
                if (X <= x1 && Y <= y1 && fast_texel<F::ROTATES>(fb, rot, atlas, X, Y, &texel)) {
                    const uint32_t a = blend ? layer_alpha(texel, blend, alpha_mod) : 255u;
                    uint32_t* px = buf + (Y - Y0) * OBS_W + X;
                    if (a == 255u) *px = texel;
                    else if (a != 0u) *px = blend_word(*px, texel, a);
                }
            }
    __syncwarp();
}

// The finished band: RGBA -> packed RGB in place (a lane reads 4 pixels and writes 3 words per round; round j's output
// [384 j, 384 j + 384) lies below every later round's input, and within a round all reads precede the writes), then ONE
// 1 536-byte TMA bulk store shared -> global (async proxy), issued by the warp that drew the band; the warp waits for the
// copy to have READ its band buffer right before it draws into the buffer again, so the drain overlaps the ticket /
// descriptor work in between.
PG2_DEV void band_store(uint8_t* __restrict__ dst, uint32_t* buf, int lane) {
    for (int j = 0; j < BAND_PX / 4 / 32; j++)
        for (int l = lane; l < 32; l += WARP_LANES) {
            const int g = j * 32 + l;
            const Word16 w = ((const Word16*)buf)[g];
            __syncwarp();
            buf[3 * g] = byte_perm(w.a, w.b, 0x4210u);
            buf[3 * g + 1] = byte_perm(w.b, w.c, 0x5421u);
            buf[3 * g + 2] = byte_perm(w.c, w.d, 0x6542u);
        }
#ifdef PG2_HOSTSIM
    memcpy(dst, buf, BAND_BYTES);
#else
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy smem writes -> async proxy
    __syncwarp();
    if (lane == 0) {
        uint32_t src = (uint32_t)__cvta_generic_to_shared(buf);
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "n"(BAND_BYTES) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
#endif
}

// Draw the frame: warps take bands from a ticket counter (a warp that drew cheap bands simply takes more of them),
// per band: base pass, post blits in submission order, bulk store.
// cache_img != nullptr (G::STATIC_VIEW): the env's base image; f.reuse says whether to load it or to (draw and) store it.
template <class G, class F>
PG2_DEV_NOINLINE void frame_rasterise(F& f, const uint32_t* __restrict__ atlas, uint8_t* __restrict__ dst, uint8_t* __restrict__ cache_img = nullptr) {
    const int lane = threadIdx.x % WARP_LANES, warp = threadIdx.x / WARP_LANES % (RENDER_THREADS / 32);
    uint32_t* buf = f.band_px[warp];
    const int npost = f.npost;
    for (;;) {
        int band = 0;
        if (lane == 0) { band = smem_atomic_inc(&f.next_band); frame_store_wait(); }   // the previous band has left the buffer
        band = warp_bcast(band);
        if (band >= NUM_BANDS) break;
        if (cache_img != nullptr && f.reuse) {
            band_from_cache(f, warp, buf, cache_img + band * BAND_CACHE_BYTES, lane);
        } else {
            raster_band_base<G>(f, atlas, band, lane, buf);
            if (cache_img != nullptr) { __syncwarp(); band_to_cache(buf, cache_img + band * BAND_CACHE_BYTES, lane); }
        }
        __syncwarp();
        for (int base = 0; base < npost; base += 32) {
            uint32_t m = 0u;
            for (int l = lane; l < 32; l += WARP_LANES) {
                const int k = base + l;
                m |= lane_ballot(k < npost && (f.bandmask[k < npost ? k : 0] >> band & 1u), l);
            }
            while (m) {
                const int k = base + __ffs(m) - 1;
                m &= m - 1u;
                draw_blit_band(f, atlas, k, band * BAND_ROWS, lane, buf);
            }
        }
        band_store(dst + band * BAND_BYTES, buf, lane);
    }
}

// Per-CTA table of the game's tile textures (ids < MAX_TILE_TEX) as window cell words, filled once before the first frame.
template <class G, class F>
PG2_DEV void frame_init_tiletex(F& f, const TexInfo* __restrict__ tex) {
    for (int t = threadIdx.x; t < MAX_TILE_TEX; t += CTA_THREADS) {
        uint32_t w = 0u;
        if (t < G::NUM_TEX) {
            const TexInfo ti = tex[t];
            const uint32_t cls = (G::TILE_CLASSES > 1) ? (uint32_t)G::tile_class((uint32_t)t) : 0u;
            w = (ti.offset & CELL_OFFSET_MASK) | (ti.blend ? 1u << 28 : 0u) | cls << 29 | CELL_PRESENT;
        }
        f.tileword[t] = w;
    }
    for (int k = threadIdx.x; k < OBS_W; k += CTA_THREADS) f.rowcell[F::WINR * OBS_W + k] = 0u;
    for (int w = threadIdx.x; w < RENDER_THREADS / 32; w += CTA_THREADS) {
        f.mbar_phase[w] = 0u;
#ifndef PG2_HOSTSIM
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(&f.mbar[w])) : "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
#endif
    }
    __syncthreads();
}

}  // namespace pg2
