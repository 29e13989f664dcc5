/* TEST INFRASTRUCTURE. One synthetic scene of the rasteriser tests (tests/test_raster_spec.py): the camera, a background,
 * a tile map and a list of post-blit requests. Shared by the harness (harness.cu, built with nvcc and with g++), the plain
 * reference (scene_ref.c) and the Python generator, which packs the same layout with numpy (SCENE_DTYPE). */
#ifndef PG2_TEST_SCENE_H
#define PG2_TEST_SCENE_H
#include <stdint.h>

#define SC_MAX_CAND 320     /* post-blit candidates of one scene (more than two rounds of emit_post_blits) */
#define SC_MAP 64           /* tile map: SC_MAP x SC_MAP cells */
#define SC_NO_TILE 255
#define SC_NUM_TEX 64       /* texture ids: 0..15 tile class 0, 16..31 tile class 1, 32..63 backgrounds and sprites */

/* mode 0: nothing, 1: render_texture (x, y world position, scale, alpha, flip), 2: render_texture_rotated (rotation in
 * radians), 3: explicit float destination rect (x, y, w, h) + angle in degrees */
typedef struct {
    int32_t mode, tex, flip, pad;
    float x, y, w, h, scale, alpha, rotation, pad2;
    double angle;
} sc_post;

typedef struct {
    float cam_x, cam_y, cam_scale;   /* cam_scale is for a 64-pixel wide view; a human frame multiplies it by width / 64 */
    int32_t bg_tex;
    float bg_x, bg_y, bg_scale;
    int32_t map_x0, map_y0;          /* tile (x, y), render space, is map[(y - map_y0) * SC_MAP + x - map_x0] */
    int32_t outside;                 /* tile id of every cell outside the map (SC_NO_TILE: none) */
    int32_t npost, pad;
    uint8_t map[SC_MAP * SC_MAP];
    sc_post post[SC_MAX_CAND];
} sc_scene;

/* bytes of a scene that describe its base image (everything before npost) */
#define SC_BASE_BYTES (10 * 4)
#define SC_MAP_OFFSET (12 * 4)

#ifdef __CUDACC__
#define SC_FN static inline __host__ __device__
#else
#define SC_FN static inline
#endif
SC_FN int sc_tile_class(int tex, int nclass) { return nclass > 1 && tex >= 16 ? 1 : 0; }
SC_FN int sc_tile_at(const sc_scene* s, int x, int y) {
    const int mx = x - s->map_x0, my = y - s->map_y0;
    if (mx < 0 || my < 0 || mx >= SC_MAP || my >= SC_MAP) return s->outside;
    return s->map[my * SC_MAP + mx];
}

#endif
