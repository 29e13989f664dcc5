/* TEST INFRASTRUCTURE. Plain reference of a synthetic scene (scene.h): render_game's painter's order drawn with the
 * written blit specification, oracle/raster.c (pg2o_blit). Compiled with gcc -O2 -ffp-contract=off together with the
 * unchanged raster.c; shares no code with the engine's rasteriser.
 *   1. clear to (0, 0, 0, 255)
 *   2. background: render_texture
 *   3. tiles of the camera window (System_Tilemap::render), y-major, x-minor: render_texture
 *   4. post blits in submission order: mode 1 render_texture, mode 2 render_texture_rotated, mode 3 rect + angle */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../oracle/raster.h"
#include "scene.h"

typedef struct { uint32_t offset; uint16_t w, h; uint32_t blend; } ref_texinfo;   /* the engine's TexInfo layout */

typedef struct {
    const ref_texinfo* tex;
    const uint32_t* atlas;   /* R | G << 8 | B << 16 | A << 24 per texel: bytes R, G, B, A in memory */
    uint8_t* target;
    int tw, th;
    float cam_x, cam_y, cam_scale, size_x, size_y;
} ref_ctx;

static pg2o_texture texture(const ref_ctx* r, int id) {
    pg2o_texture t;
    t.w = r->tex[id].w; t.h = r->tex[id].h; t.blend = r->tex[id].blend != 0;
    t.rgba = (const uint8_t*)(r->atlas + r->tex[id].offset);
    return t;
}

/* SDL_SetTextureAlphaMod(tex, 255 * alpha): float -> Uint8 */
static uint8_t alpha_mod_of(float alpha) { return alpha != 1.0f ? (uint8_t)(int)(255.0f * alpha) : (uint8_t)255; }

/* One axis of Renderer::render_texture: world position -> destination, cull, crop a destination that starts left of /
 * above the screen, crop one that ends beyond it, pad the source by ceil(1 / (scale * camera scale)) texels and
 * compensate the destination for the padding and the fractional source start, mirror the source rect when flipped.
 * Returns 0 when the blit is culled. */
static int render_axis(float pos, float cam, float cs, float size, int tex_len, float scale, int flip, int y_axis,
                       float* src0_out, float* srcl_out, float* dst0_out, float* dstl_out) {
    float src0 = 0.0f, srcl = (float)tex_len;
    float dst0 = (pos - cam) * cs + size * 0.5f;
    float dstl = (float)tex_len * scale * cs;
    if (y_axis ? (dst0 >= size) : (dst0 > size)) return 0;
    if (dst0 + dstl < 0.0f) return 0;
    if (dst0 < 0.0f) {
        float ratio = -dst0 / dstl;
        src0 = src0 + srcl * ratio;
        srcl = srcl - src0;
        dstl = dstl + dst0;
        dst0 = 0.0f;
    }
    if (dst0 + dstl > size) {
        float ratio = (dst0 + dstl - size) / dstl;
        srcl = srcl * (1.0f - ratio);
        dstl = size - dst0;
    }
    int padding = (int)ceilf(1.0f / (scale * cs));
    int si0 = (int)floorf(src0);
    int sil = (int)ceilf(srcl) + padding;
    float offset = src0 - (float)si0;
    float size_ratio = (float)sil / srcl;
    dstl = dstl * size_ratio;
    dst0 = dst0 - offset * (dstl / srcl);
    if (flip) si0 = tex_len - sil - si0;
    *src0_out = (float)si0; *srcl_out = (float)sil; *dst0_out = dst0; *dstl_out = dstl;
    return 1;
}

/* Renderer::render_texture */
static void render_texture(const ref_ctx* r, int id, float px, float py, float scale, float alpha, int flip) {
    pg2o_texture t = texture(r, id);
    float src[4], dst[4];
    int vx = render_axis(px, r->cam_x, r->cam_scale, r->size_x, t.w, scale, flip, 0, &src[0], &src[2], &dst[0], &dst[2]);
    int vy = render_axis(py, r->cam_y, r->cam_scale, r->size_y, t.h, scale, 0, 1, &src[1], &src[3], &dst[1], &dst[3]);
    if (!vx || !vy) return;
    pg2o_blit(r->target, r->tw, r->th, &t, src, dst, 0.0, flip ? 1 : 0, alpha_mod_of(alpha));
}

/* Renderer::render_texture_rotated: the whole texture, no culling or cropping; angle = rotation * 180 / pi */
static void render_texture_rotated(const ref_ctx* r, int id, float px, float py, float rotation, float scale, float alpha) {
    pg2o_texture t = texture(r, id);
    float dst[4];
    dst[0] = (px - r->cam_x) * r->cam_scale + r->size_x * 0.5f;
    dst[1] = (py - r->cam_y) * r->cam_scale + r->size_y * 0.5f;
    dst[2] = (float)t.w * scale * r->cam_scale;
    dst[3] = (float)t.h * scale * r->cam_scale;
    double angle = (double)(rotation * 180.0f) / 3.14159265358979323846;
    pg2o_blit(r->target, r->tw, r->th, &t, NULL, dst, angle, 0, alpha_mod_of(alpha));
}

/* System_Tilemap::render's window: inclusive tile index range */
static void tile_window(const ref_ctx* r, int* lx, int* ly, int* ux, int* uy) {
    float hx = r->size_x * 0.5f / r->cam_scale, hy = r->size_y * 0.5f / r->cam_scale;
    float ax = (r->cam_x - hx) * (1.0f / 16.0f), ay = (r->cam_y - hy) * (1.0f / 16.0f);
    float aw = r->size_x * (1.0f / 16.0f) / r->cam_scale, ah = r->size_y * (1.0f / 16.0f) / r->cam_scale;
    *lx = (int)floorf(ax); *ly = (int)floorf(ay);
    *ux = (int)ceilf(ax + aw); *uy = (int)ceilf(ay + ah);
}

/* out: width x height x 3 (RGB). nclass: tile shape classes of the trait set (0: no tile layer). */
void scene_ref_render(const sc_scene* s, const void* texinfo, const uint32_t* atlas, int nclass, int width, int height, uint8_t* out) {
    ref_ctx r;
    r.tex = (const ref_texinfo*)texinfo; r.atlas = atlas;
    r.tw = width; r.th = height;
    r.size_x = (float)width; r.size_y = (float)height;
    r.cam_x = s->cam_x; r.cam_y = s->cam_y; r.cam_scale = s->cam_scale * r.size_x / 64.0f;
    r.target = (uint8_t*)malloc((size_t)width * height * 4);
    for (size_t p = 0; p < (size_t)width * height; p++) { r.target[4 * p] = 0; r.target[4 * p + 1] = 0; r.target[4 * p + 2] = 0; r.target[4 * p + 3] = 255; }
    render_texture(&r, s->bg_tex, s->bg_x, s->bg_y, s->bg_scale, 1.0f, 0);
    if (nclass > 0) {
        int lx, ly, ux, uy;
        tile_window(&r, &lx, &ly, &ux, &uy);
        for (int y = ly; y <= uy; y++)
            for (int x = lx; x <= ux; x++) {
                int t = sc_tile_at(s, x, y);
                if (t == SC_NO_TILE) continue;
                render_texture(&r, t, (float)x * 16.0f, (float)y * 16.0f, 16.0f / (float)r.tex[t].w, 1.0f, 0);
            }
    }
    for (int k = 0; k < s->npost && k < SC_MAX_CAND; k++) {
        const sc_post* p = &s->post[k];
        if (p->mode == 1) render_texture(&r, p->tex, p->x, p->y, p->scale, p->alpha, p->flip != 0);
        else if (p->mode == 2) render_texture_rotated(&r, p->tex, p->x, p->y, p->rotation, p->scale, p->alpha);
        else if (p->mode == 3) {
            pg2o_texture t = texture(&r, p->tex);
            float dst[4] = { p->x, p->y, p->w, p->h };
            pg2o_blit(r.target, r.tw, r.th, &t, NULL, dst, p->angle, 0, 255);
        }
    }
    for (size_t q = 0; q < (size_t)width * height; q++) { out[3 * q] = r.target[4 * q]; out[3 * q + 1] = r.target[4 * q + 1]; out[3 * q + 2] = r.target[4 * q + 2]; }
    free(r.target);
}
