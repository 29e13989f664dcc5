// Climber — device restatement of /root/reference/games/climber/:
//   step logic  cenv_step climber.cpp:323-372; System_Agent::update common_systems.cpp:184-270;
//               System_Mob_AI::update :109-168; System_Point::update :66-107;
//               System_Sprite_Render::update :8-40; System_Tilemap::get_collision tilemap.cpp:199-260
//   level gen   System_Tilemap::regenerate tilemap.cpp:75-172 (+ spawn helpers :40-73), reset() climber.cpp:459-494
//   frame       render_game climber.cpp:431-457; tilemap.cpp:174-197; common_systems.cpp:42-64, 272-296
// Compile-time mode of the reference: easy_mode = false (tilemap.h:33).
#pragma once
#include "../pg2_common.cuh"
#include "../pg2_render.cuh"
#include "../pg2_state.cuh"
#include "../pg2_tilecoll.cuh"
#include "../pg2_uset.cuh"
#include "../pg2_warp.cuh"
#include "platform_bgs.h"

namespace pg2 {

// Entity pools are slot-major: field[slot * N + env]. Slot = entity id (creation order).
#define PG2_CLIMBER_FIELDS(F)                                                                  \
    PG2_ENV_MAJOR(F)(uint8_t, tiles, 1280) /* [y + x*64], 20 x 64 */                            \
    F(int32_t, num_ents, 1)                                                                     \
    F(uint8_t, ent_type, 40)    /* 1 mob, 2 point, 0 destroyed */                               \
    F(float, ent_x, 40)                                                                         \
    F(float, ent_y, 40)                                                                         \
    F(float, ent_vx, 40)        /* Component_Mob_AI::velocity_x */                              \
    F(int32_t, ent_spawn_x, 40)                                                                 \
    F(float, ent_anim_t, 40)                                                                    \
    F(uint8_t, ent_frame, 40)                                                                   \
    F(uint8_t, ent_flip, 40)                                                                    \
    F(uint8_t, sprite_order, 40) /* iteration order of System_Sprite_Render::entities at reset */ \
    F(int32_t, nb_sprite, 1)    /* persisted bucket count (Q25) */                              \
    F(float, ax, 1) F(float, ay, 1) F(float, avx, 1) F(float, avy, 1)                           \
    F(uint8_t, on_ground, 1) F(uint8_t, face_forward, 1) F(float, agent_t, 1)                   \
    F(int32_t, bg_index, 1) F(float, bg_offset, 1) F(int32_t, agent_theme, 1) F(int32_t, map_theme, 1)

PG2_DEFINE_STATE(ClimberState, PG2_CLIMBER_FIELDS)

struct Climber {
    using State = ClimberState;
    static constexpr int W = 20, H = 64, MAX_ENTS = 40;
    static constexpr int SUB_STEPS = 4;
    static constexpr bool LANE_AWARE = true;    // step(): per-entity loops are strided over ctx's lanes
    static constexpr int STEP_LANES = 32;       // lanes per environment in k_step
    static constexpr int MAX_POST = 48;        // capacity of the frame's post-blit list
    static constexpr bool ROTATES = false;     // some blits are rotated
    static constexpr bool SLOW_RESET = false;   // level generation is long: run it concurrently with the render of the other envs
    static constexpr int RESET_ARENA = 4 * 1024;   // per-warp level-generation scratch (high water measured with PG2_ARENA_TRACE)
    static constexpr bool PREFETCH_LEVELS = true;    // the RNG is only drawn inside reset(): the next level is generated one episode ahead (+8 % at 4096 envs)
    static constexpr int PREFETCH_MIN_EPISODE = 0;   // level prefetch whatever max_episode_steps is
    static const char* reset_keeps() { return " cam_y "; }   // fields reset() does not write (they persist across episodes)
    static constexpr int TILE_CLASSES = 2;   // wall_mid textures are 64x64, one wall_top texture is 64x53
    static constexpr int WIN_ROWS = 23;        // most tile rows the camera window can span (zoom-dependent; frame table sizing)
    static constexpr int BLIT_UNROLL = 1;     // post-blit patches fetched together (pg2_render.cuh draw_blit_band)
    static constexpr int RENDER_MIN_CTAS = 8;   // CTAs per SM the register allocation of k_render aims at
    static constexpr int DEFAULT_MODE = 1;    // distribution mode the reference compiles in (tilemap.h Config): 0 easy, 1 hard, 2 memory / extreme
    static bool mode_supported(int mode) { return mode == 0 || mode == 1; }
    static constexpr bool HAS_TILES = true;     // the frame has a tile layer
    static constexpr bool STATIC_VIEW = false;   // the camera follows the agent: the base image changes every frame (a camera-keyed cache measured slower)
    enum Tile { EMPTY = 0, WALL_TOP, WALL_MID };
    enum Ent { E_NONE = 0, E_MOB, E_POINT };
    enum Tex {
        T_WALL_TOP0 = 0, T_WALL_MID0 = 4, T_ENEMY0 = 8, T_CRYSTAL = 10,
        T_AGENT0 = 11,   // 4 themes x {stand, jump(walk4), walk1, walk2}
        T_BG0 = 27, NUM_TEX = 27 + PG2_NUM_PLATFORM_BACKGROUNDS
    };

    static const char* const* texture_names(int* count) {
        static const char* const names[NUM_TEX] = {
            "assets/platformer/tileBlue_05.png", "assets/platformer/tileGreen_05.png",
            "assets/platformer/tileYellow_06.png", "assets/platformer/tileBrown_06.png",
            "assets/platformer/tileBlue_08.png", "assets/platformer/tileGreen_08.png",
            "assets/platformer/tileYellow_09.png", "assets/platformer/tileBrown_09.png",
            "assets/platformer/enemySwimming_1.png", "assets/platformer/enemySwimming_2.png",
            "assets/misc_assets/yellowCrystal.png",
            "assets/platformer/playerBlue_stand.png", "assets/platformer/playerBlue_walk4.png",
            "assets/platformer/playerBlue_walk1.png", "assets/platformer/playerBlue_walk2.png",
            "assets/platformer/playerGreen_stand.png", "assets/platformer/playerGreen_walk4.png",
            "assets/platformer/playerGreen_walk1.png", "assets/platformer/playerGreen_walk2.png",
            "assets/platformer/playerGrey_stand.png", "assets/platformer/playerGrey_walk4.png",
            "assets/platformer/playerGrey_walk1.png", "assets/platformer/playerGrey_walk2.png",
            "assets/platformer/playerRed_stand.png", "assets/platformer/playerRed_walk4.png",
            "assets/platformer/playerRed_walk1.png", "assets/platformer/playerRed_walk2.png",
            PG2_PLATFORM_BACKGROUNDS
        };
        *count = NUM_TEX;
        return names;
    }

    // System_Tilemap::get (tilemap.h:66-71): out of bounds is wall_mid. (x, y) in map space.
    static PG2_DEV int get(const uint8_t* tiles, int x, int y) {
        if (x < 0 || y < 0 || x >= W || y >= H) return WALL_MID;
        return tiles[y + x * H];
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV_NOINLINE bool step(const State& s, const CommonState& c, int env, int action, float* reward, const StepCtx& ctx) {
        const int N = s.N;
        const uint8_t* tiles = s.tiles + (size_t)env * (W * H);
        const float dt = 1.0f / SUB_STEPS;
        const int nents = s.num_ents[env];
        auto tile_at = [&](int x, int y) { return get(tiles, x, H - 1 - y); };
        auto wall = [](int id) { return (id == WALL_MID || id == WALL_TOP) ? COLL_FULL : COLL_NONE; };

        float ax = s.ax[env], ay = s.ay[env], avx = s.avx[env], avy = s.avy[env], agent_t = s.agent_t[env];
        bool on_ground = s.on_ground[env] != 0, face_forward = s.face_forward[env] != 0;
        float cam_y = c.cam_y[env];

        const float max_jump = 1.55f, gravity = 0.2f, max_speed = 0.5f, mix = 0.2f, air_control = 0.15f;
        const float movement_x = (float)((action == 6 || action == 7 || action == 8) - (action == 0 || action == 1 || action == 2));
        const bool jump = (action == 2 || action == 5 || action == 8);

        bool dead = false;
        int point_delta = 0, points_available = 0;
        for (int ss = 0; ss < SUB_STEPS; ss++) {
            // ---- System_Agent::update
            {
                float mix_x = on_ground ? mix : __fmul_rn(mix, air_control);
                avx = __fadd_rn(avx, __fmul_rn(__fmul_rn(mix_x, __fsub_rn(__fmul_rn(max_speed, movement_x), avx)), dt));
                if (fabsf(avx) < __fmul_rn(__fmul_rn(mix_x, max_speed), dt)) avx = 0.0f;
                if (jump && on_ground) avy = -max_jump;
                avy = __fadd_rn(avy, __fmul_rn(gravity, dt));
                if (fabsf(avy) > max_jump) avy = __fmul_rn(avy > 0.0f ? 1.0f : -1.0f, max_jump);
                ax = __fadd_rn(ax, __fmul_rn(avx, dt));
                ay = __fadd_rn(ay, __fmul_rn(avy, dt));
                Rect world{ __fadd_rn(ax, -0.5f), __fadd_rn(ay, -1.0f), 1.0f, 1.0f };
                CollisionResult cd = tile_collision(world, tile_at, wall, false, 0.0f, &ctx);
                float dpx = __fsub_rn(cd.x, world.x), dpy = __fsub_rn(cd.y, world.y);
                on_ground = dpy < 0.0f && cd.collided;
                ax = __fsub_rn(cd.x, -0.5f);
                ay = __fsub_rn(cd.y, -1.0f);
                if (dpx != 0.0f) avx = 0.0f;
                if (on_ground) avy = 0.0f;
                cam_y = __fmul_rn(__fsub_rn(__fsub_rn(ay, 8.0f), 0.5f), UNIT_TO_PIXELS);
                agent_t = __fadd_rn(agent_t, __fmul_rn(0.1f, dt));
                agent_t = fmodf(agent_t, 1.0f);
                if (movement_x > 0.0f) face_forward = true;
                else if (movement_x < 0.0f) face_forward = false;
            }
            const Rect agent_rect{ __fadd_rn(-0.5f, ax), __fadd_rn(-1.0f, ay), 1.0f, 1.0f };

            // ---- System_Mob_AI::update, System_Point::update, System_Sprite_Render::update (animation)
            bool hit = false;
            int delta = 0, avail = 0;
            for (int e = ctx.lane; e < nents; e += ctx.nlanes) {
                int type = s.ent_type[e * N + env];
                if (type == E_MOB) {
                    float x = s.ent_x[e * N + env], y = s.ent_y[e * N + env], vx = s.ent_vx[e * N + env];
                    // fetched here, before the first store of the entity (stores cannot be proven not to alias later loads)
                    const int spawn_x = s.ent_spawn_x[e * N + env], frame0 = s.ent_frame[e * N + env];
                    const float anim_t0 = s.ent_anim_t[e * N + env];
                    x = __fadd_rn(x, __fmul_rn(vx, dt));
                    Rect wall_sensor{ __fsub_rn(x, 0.5f), __fsub_rn(y, 0.6f), 1.0f, 0.5f };
                    CollisionResult wc = tile_collision(wall_sensor, tile_at, wall);
                    x = __fadd_rn(wc.x, 0.5f);
                    Rect rect{ __fadd_rn(-0.4f, x), __fadd_rn(-0.4f, y), 0.8f, 0.8f };
                    if (check_collision(agent_rect, rect)) hit = true;
                    bool end_patrol = x > (float)(spawn_x + 4) || x < (float)(spawn_x - 4);
                    if (wc.collided || end_patrol) vx = __fmul_rn(vx, -1.0f);
                    s.ent_x[e * N + env] = x; s.ent_vx[e * N + env] = vx;
                    s.ent_flip[e * N + env] = vx < 0.0f;
                    // System_Sprite_Render::update (animation) of the same entity
                    float t = __fadd_rn(anim_t0, dt);
                    int adv = f2i(__fmul_rn(t, 0.2f));
                    t = __fsub_rn(t, __fdiv_rn((float)adv, 0.2f));
                    s.ent_anim_t[e * N + env] = t;
                    s.ent_frame[e * N + env] = (uint8_t)((frame0 + adv) % 2);
                } else if (type == E_POINT) {
                    Rect rect{ __fadd_rn(-0.5f, s.ent_x[e * N + env]), __fadd_rn(-0.5f, s.ent_y[e * N + env]), 1.0f, 1.0f };
                    if (check_collision(agent_rect, rect)) { delta++; s.ent_type[e * N + env] = E_NONE; }
                    else avail++;
                }
            }
            dead = ctx.any(hit);
            point_delta = ctx.sum(delta);
            points_available = ctx.sum(avail);
            if (dead || points_available == 0) break;
        }

        if (ctx.leader()) {
            s.ax[env] = ax; s.ay[env] = ay; s.avx[env] = avx; s.avy[env] = avy; s.agent_t[env] = agent_t;
            s.on_ground[env] = on_ground; s.face_forward[env] = face_forward;
            c.cam_y[env] = cam_y;
            c.sprites_valid[env] = 1;
        }
        *reward = __fadd_rn((float)point_delta, __fmul_rn((float)(points_available == 0), 10.0f));
        return dead || points_available == 0;
    }

    // ---------------------------------------------------------------------------------------
    struct Gen {
        uint8_t* tiles;
        WarpCtx* w;
        PG2_DEV void set(int x, int y, int id) { if (x < 0 || y < 0 || x >= W || y >= H) return; tiles[y + x * H] = (uint8_t)id; }
        PG2_DEV_NOINLINE void set_area(int x, int y, int width, int height, int id) {
            if (width > 0 && height > 0)
                for (int i = w->lane; i < width * height; i += WARP_LANES) set(x + i / height, y + i % height, id);
            __syncwarp();
        }
        PG2_DEV_NOINLINE void set_area_with_top(int x, int y, int width, int height, int mid, int top) {
            set_area(x, y, width, height - 1, mid);
            set_area(x, y + height - 1, width, 1, top);
        }
    };

    static PG2_DEV_NOINLINE void regenerate(const State& s, const CommonState& c, int env, WarpCtx& w) {
        const int N = s.N, lane = w.lane;
        uint8_t* tiles = w.alloc<uint8_t>(W * H);
        uint8_t* etype = w.alloc<uint8_t>(MAX_ENTS);
        float* ex = w.alloc<float>(MAX_ENTS);
        float* ey = w.alloc<float>(MAX_ENTS);
        float* evx = w.alloc<float>(MAX_ENTS);
        int* espawn = w.alloc<int>(MAX_ENTS);
        int* candidates = w.alloc<int>(16);
        int nents = 0;
        bool overflow = false;
        Gen g{ tiles, &w };
        w.fill<uint8_t>(tiles, W * H, 0);
        g.set_area_with_top(0, 0, W, 1, WALL_MID, WALL_TOP);
        g.set_area(0, 0, 1, H, WALL_MID);
        g.set_area(W - 1, 0, 1, H, WALL_MID);
        g.set_area(0, H - 1, W, 1, WALL_MID);

        auto spawn = [&](int type, int x, int y, float vx) {
            if (nents >= MAX_ENTS) { overflow = true; return; }
            etype[nents] = (uint8_t)type;
            ex[nents] = __fadd_rn((float)x, 0.5f);
            ey[nents] = __fadd_rn((float)(H - 1 - y), 0.5f);
            evx[nents] = vx; espawn[nents] = x;
            nents++;
        };

        int difficulty = w.rng.uniform_int(1, 3);
        int num_platforms = w.rng.uniform_int(difficulty * difficulty + 1, (difficulty + 1) * (difficulty + 1) + 1);
        int curr_x = w.rng.uniform_int(2, W - 3);
        int curr_y = 1;
        const int margin_x = 3;
        const float enemy_prob = w.mode == 0 ? 0.2f : 0.5f;   // cfg.easy_mode ? .2 : .5 (tilemap.cpp:118)
        const float max_dyf = __fdiv_rn(__fmul_rn(1.5f, 1.5f), __fmul_rn(2.0f, 0.2f));
        const int max_dy = f2i(__fsub_rn(max_dyf, 0.5f));

        for (int platform = 0; platform < num_platforms; platform++) {
            int delta_y = w.rng.uniform_int(3, max_dy - 1);
            bool can_spawn_enemy = (curr_x >= margin_x) && (curr_x <= W - 1 - margin_x);
            if (can_spawn_enemy && (w.rng.uniform_real(0.0f, 1.0f) < enemy_prob)) {
                int y = curr_y + w.rng.uniform_int(0, 1) + 2;
                float vx = __fmul_rn(0.15f, __fsub_rn(__fmul_rn((float)w.rng.uniform_int(0, 1), 2.0f), 1.0f));
                spawn(E_MOB, curr_x, y, vx);
            }
            curr_y += delta_y;
            int plat_len = 2 + w.rng.uniform_int(0, 9);
            int vx = w.rng.uniform_int(0, 1) * 2 - 1;
            if (curr_x < margin_x) vx = 1;
            if (curr_x > W - margin_x) vx = -1;
            int ncand = 0;
            __syncwarp();
            for (int j = 0; j < plat_len; j++) {
                int nx = curr_x + (j + 1) * vx;
                if (nx <= 0 || nx >= W - 1) break;
                candidates[ncand++] = nx;
                g.set(nx, curr_y, WALL_TOP);   // set_area_with_top(nx, curr_y, 1, 1, ...) == one wall_top cell
            }
            __syncwarp();
            if (ncand == 0) { if (lane == 0) c.fault[env] |= 2; ncand = 1; candidates[0] = curr_x; }   // Q20: never hit
            bool want_point = w.rng.uniform_real(0.0f, 1.0f) < 0.5f;
            if (want_point || platform == num_platforms - 1) {
                int point_x = candidates[w.rng.uniform_int(0, ncand - 1)];
                spawn(E_POINT, point_x, curr_y + 1, 0.0f);
            }
            curr_x = candidates[w.rng.uniform_int(0, ncand - 1)];
            __syncwarp();
        }

        // ---- reset() tail (climber.cpp:464-493)
        int bg_index = w.rng.uniform_int(0, PG2_NUM_PLATFORM_BACKGROUNDS - 1);
        float bg_offset = w.rng.uniform_real(0.0f, 1.0f);
        int agent_theme = w.rng.uniform_int(0, 3);
        int map_theme = w.rng.uniform_int(0, 3);

        // iteration order of System_Sprite_Render::entities (every mob and point, ids ascending)
        USet<MAX_ENTS, 64>* us = w.alloc<USet<MAX_ENTS, 64>>(1);
        uint8_t* order = w.alloc<uint8_t>(MAX_ENTS);
        __syncwarp();
        us->init(s.nb_sprite[env]);
        for (int e = 0; e < nents; e++) us->insert(e);
        int n_sprite = us->order(order);
        int nb_sprite = us->nb;
        __syncwarp();
        for (int k = lane; k < n_sprite; k += WARP_LANES) s.sprite_order[k * N + env] = order[k];

        uint8_t* gt = s.tiles + (size_t)env * (W * H);
        for (int i = lane; i < W * H / 4; i += WARP_LANES) ((uint32_t*)gt)[i] = ((const uint32_t*)tiles)[i];
        for (int e = lane; e < nents; e += WARP_LANES) {
            s.ent_type[e * N + env] = etype[e];
            s.ent_x[e * N + env] = ex[e]; s.ent_y[e * N + env] = ey[e];
            s.ent_vx[e * N + env] = evx[e]; s.ent_spawn_x[e * N + env] = espawn[e];
            s.ent_anim_t[e * N + env] = 0.0f; s.ent_frame[e * N + env] = 0; s.ent_flip[e * N + env] = 0;
        }
        if (lane == 0) {
            s.num_ents[env] = nents;
            s.nb_sprite[env] = nb_sprite;
            s.ax[env] = 1.5f;
            s.ay[env] = __fadd_rn((float)(H - 2), 1.0f);
            s.avx[env] = 0.0f; s.avy[env] = 0.0f;
            s.on_ground[env] = 0; s.face_forward[env] = 1; s.agent_t[env] = 0.0f;
            s.bg_index[env] = bg_index; s.bg_offset[env] = bg_offset;
            s.agent_theme[env] = agent_theme; s.map_theme[env] = map_theme;
            c.cam_x[env] = __fmul_rn(__fdiv_rn((float)W, 2.0f), UNIT_TO_PIXELS);
            c.sprites_valid[env] = 0;
            if (overflow) c.fault[env] |= 1;
        }
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV int tile_class(uint32_t tex) { return tex < (uint32_t)T_WALL_MID0 ? 1 : 0; }

    template <class F>
    static PG2_DEV_NOINLINE void build_frame(const State& s, const CommonState& c, int env, F& f, const TexInfo* tex) {
        const int N = s.N;
        Camera cam{ c.cam_x[env], c.cam_y[env], __fdiv_rn(__fmul_rn(0.2f, f.view_w), 64.0f), f.view_w, f.view_h };
        int lx, ly, ux, uy;
        tile_window(cam, &lx, &ly, &ux, &uy);
        const int ncol = min(ux - lx + 1, MAX_WIN), nrow = min(uy - ly + 1, MAX_WIN);
        const int nents = s.num_ents[env];
        const bool sprites = c.sprites_valid[env] != 0;
        const int theme = s.map_theme[env];
        // background (e.g. maze.cpp:402-408): the blit itself is built by build_tile_layer below
        const int bg = T_BG0 + s.bg_index[env];
        const TexInfo bt = tex[bg];
        const float bg_x = __fmul_rn(-s.bg_offset[env], __fsub_rn(__fdiv_rn((float)bt.w, (float)bt.h), 1.0f));
        const float bg_scale = __fdiv_rn(__fmul_rn(64.0f, UNIT_TO_PIXELS), (float)bt.h);
        // live sprites in set order; destroyed points simply drop out of the (order-preserving) set
        const int nlive = live_list(f, sprites ? nents : 0, [&](int j) {
            const int e = s.sprite_order[j * N + env];
            return s.ent_type[e * N + env] != E_NONE ? e : -1; });
        // tile layer: class 0 = wall_mid texture of the theme, class 1 = wall_top texture
        const uint8_t* tiles = s.tiles + (size_t)env * (W * H);
        build_tile_layer(f, cam, tex, 2, lx, ly, ncol, nrow, [&](int cls) { return (cls ? T_WALL_TOP0 : T_WALL_MID0) + theme; }, [&](int x, int y) {
            const int id = get(tiles, x, H - 1 - y);
            return id == WALL_MID ? T_WALL_MID0 + theme : id == WALL_TOP ? T_WALL_TOP0 + theme : (int)NO_TILE;
        }, bg, bg_x, 0.0f, bg_scale);
        emit_post_blits(f, tex, nlive + 1, [&](int k, BlitReq& b, BlitRot&) {
            if (k < nlive) {
                const int e = f.live[sort_perm(nlive, k)];
                int type = s.ent_type[e * N + env];
                int t = type == E_POINT ? T_CRYSTAL : T_ENEMY0 + s.ent_frame[e * N + env];
                float off = type == E_POINT ? -0.5f : -0.4f;
                float px = __fmul_rn(__fadd_rn(s.ent_x[e * N + env], off), UNIT_TO_PIXELS);
                float py = __fmul_rn(__fadd_rn(s.ent_y[e * N + env], off), UNIT_TO_PIXELS);
                float sc = __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, 1.0f), UNIT_TO_PIXELS), (float)tex[t].w);
                b.plain(t, px, py, cam, sc, 1.0f, s.ent_flip[e * N + env] != 0);
            } else {
                float avx = s.avx[env];
                bool on_ground = s.on_ground[env] != 0;
                int pose = (fabsf(avx) < 0.01f && on_ground) ? 0 : (!on_ground ? 1 : (s.agent_t[env] > 0.5f ? 3 : 2));
                int t = T_AGENT0 + 4 * s.agent_theme[env] + pose;
                float px = __fmul_rn(__fsub_rn(s.ax[env], 0.5f), UNIT_TO_PIXELS);
                float py = __fmul_rn(__fsub_rn(s.ay[env], 1.0f), UNIT_TO_PIXELS);
                b.plain(t, px, py, cam, __fdiv_rn(__fmul_rn(0.8f, UNIT_TO_PIXELS), (float)tex[t].w), 1.0f, s.face_forward[env] == 0);
            }
        });
    }
};

}  // namespace pg2
