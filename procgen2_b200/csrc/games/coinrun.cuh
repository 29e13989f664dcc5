// CoinRun — device restatement of /root/reference/games/coinrun/:
//   step logic  cenv_step coinrun.cpp:341-391; System_Mob_AI::update common_systems.cpp:65-105;
//               System_Agent::update :121-252; System_Particles::update :284-313;
//               System_Sprite_Render::update :7-39; System_Tilemap::get_collision tilemap.cpp:323-396
//   level gen   System_Tilemap::regenerate tilemap.cpp:97-292 (+ spawn helpers :52-95), reset() coinrun.cpp:472-507
//   frame       render_game coinrun.cpp:443-470; tilemap.cpp:294-321; common_systems.cpp:41-63, 254-278, 315-337
// Compile-time mode of the reference: easy_mode = false, all allow_* = true (tilemap.h:40-46). easy_mode only feeds
// `allow_monsters` (tilemap.cpp:148), which nothing reads: the "easy" distribution mode generates the same levels.
#pragma once
#include "../pg2_common.cuh"
#include "../pg2_render.cuh"
#include "../pg2_state.cuh"
#include "../pg2_tilecoll.cuh"
#include "../pg2_uset.cuh"
#include "../pg2_warp.cuh"
#include "platform_bgs.h"

namespace pg2 {

// Entity pools are slot-major: field[slot * N + env] (coalesced across a warp of envs).
#define PG2_COINRUN_FIELDS(F)                                                                  \
    PG2_ENV_MAJOR(F)(uint8_t, tiles, 4096) /* [y + x*64]: Tile_ID | crate_type << 4 */         \
    F(int32_t, num_ents, 1)     /* entities created by regenerate (saws, mobs, coin) */         \
    F(uint8_t, ent_type, 40)    /* 1 saw, 2 mob, 3 coin */                                      \
    F(float, ent_x, 40)                                                                         \
    F(float, ent_y, 40)                                                                         \
    F(float, ent_vx, 40)        /* Component_Mob_AI::velocity_x */                              \
    F(float, ent_anim_t, 40)    /* Component_Animation::t */                                    \
    F(uint8_t, ent_frame, 40)   /* Component_Animation::frame_index */                          \
    F(uint8_t, ent_kind, 40)    /* walking_enemies index */                                     \
    F(uint8_t, ent_flip, 40)    /* Component_Sprite::flip_x */                                  \
    F(float, part_x, 400)       /* Component_Particles: [(slot*10 + i) * N + env] */            \
    F(float, part_y, 400)                                                                       \
    F(float, part_life, 400)                                                                    \
    F(float, part_timer, 40)    /* spawn_timer */                                               \
    F(uint8_t, sprite_order, 40) /* iteration order of System_Sprite_Render::entities */        \
    F(int32_t, num_mobs, 1)                                                                     \
    F(uint8_t, mob_order, 40)   /* iteration order of System_Particles::entities (mob ids) */   \
    F(int32_t, nb_sprite, 1)    /* persisted bucket counts of those two sets (Q25) */           \
    F(int32_t, nb_mob, 1)                                                                       \
    F(float, ax, 1)                                                                             \
    F(float, ay, 1)                                                                             \
    F(float, avx, 1)                                                                            \
    F(float, avy, 1)                                                                            \
    F(uint8_t, on_ground, 1)                                                                    \
    F(uint8_t, face_forward, 1)                                                                 \
    F(float, agent_t, 1)                                                                        \
    F(int32_t, bg_index, 1)                                                                     \
    F(float, bg_offset, 1)                                                                      \
    F(int32_t, agent_theme, 1)                                                                  \
    F(int32_t, map_theme, 1)

PG2_DEFINE_STATE(CoinRunState, PG2_COINRUN_FIELDS)

struct CoinRun {
    using State = CoinRunState;
    static constexpr int W = 64, H = 64, MAX_ENTS = 40, NPART = 10;
    static constexpr int SUB_STEPS = 4;
    static constexpr bool LANE_AWARE = true;    // step(): per-entity loops are strided over ctx's lanes
    static constexpr int STEP_LANES = 32;       // lanes per environment in k_step
    static constexpr int MAX_POST = 192;        // capacity of the frame's post-blit list
    static constexpr bool ROTATES = false;     // some blits are rotated
    static constexpr bool SLOW_RESET = false;   // level generation is long: run it concurrently with the render of the other envs
    static constexpr int RESET_ARENA = 8 * 1024;   // per-warp level-generation scratch (high water measured with PG2_ARENA_TRACE)
    static constexpr bool PREFETCH_LEVELS = true;    // the RNG is only drawn inside reset(): the next level is generated one episode ahead (+11 % at 4096 envs)
    static constexpr int PREFETCH_MIN_EPISODE = 256;   // ... unless episodes are truncated shorter than this: 12 KB of state to swap per reset then costs more than the inline reset (-7 % at 32 768 envs x 32 steps)
    static const char* reset_keeps() { return " cam_x cam_y "; }   // fields reset() does not write (they persist across episodes)
    static constexpr int TILE_CLASSES = 1;
    static constexpr int WIN_ROWS = 16;        // most tile rows the camera window can span (zoom-dependent; frame table sizing)
    static constexpr int BLIT_UNROLL = 1;     // post-blit patches fetched together (pg2_render.cuh draw_blit_band)
    static constexpr int RENDER_MIN_CTAS = 7;   // CTAs per SM the register allocation of k_render aims at
    static constexpr int DEFAULT_MODE = 1;    // distribution mode the reference compiles in (tilemap.h Config): 0 easy, 1 hard, 2 memory / extreme
    static bool mode_supported(int mode) { return mode == 0 || mode == 1; }
    static constexpr bool HAS_TILES = true;     // the frame has a tile layer
    static constexpr bool STATIC_VIEW = false;   // the camera follows the agent: the base image changes every frame (a camera-keyed cache measured slower)
    enum Tile { EMPTY = 0, WALL_TOP, WALL_MID, LAVA_TOP, LAVA_MID, CRATE };
    enum Ent { E_NONE = 0, E_SAW, E_MOB, E_COIN };
    enum Tex {
        T_WALL_TOP0 = 0,    // 6 themes "<theme>Mid.png"
        T_WALL_MID0 = 6,    // 6 themes "<theme>Center.png"
        T_LAVA_TOP = 12, T_LAVA_MID = 13,
        T_CRATE0 = 14,      // 4 crate types
        T_ENEMY0 = 18,      // 9 walking enemies x {stand, move}
        T_SAW0 = 36,        // sawHalf, sawHalf_move
        T_COIN = 38,
        T_AGENT0 = 39,      // 5 themes x {stand, jump, walk1, walk2}
        T_PARTICLE = 59,
        T_BG0 = 60,
        NUM_TEX = 60 + PG2_NUM_PLATFORM_BACKGROUNDS
    };

    static const char* const* texture_names(int* count) {
        static const char* const names[NUM_TEX] = {
            "assets/kenney/Ground/Dirt/dirtMid.png", "assets/kenney/Ground/Grass/grassMid.png", "assets/kenney/Ground/Planet/planetMid.png",
            "assets/kenney/Ground/Sand/sandMid.png", "assets/kenney/Ground/Snow/snowMid.png", "assets/kenney/Ground/Stone/stoneMid.png",
            "assets/kenney/Ground/Dirt/dirtCenter.png", "assets/kenney/Ground/Grass/grassCenter.png", "assets/kenney/Ground/Planet/planetCenter.png",
            "assets/kenney/Ground/Sand/sandCenter.png", "assets/kenney/Ground/Snow/snowCenter.png", "assets/kenney/Ground/Stone/stoneCenter.png",
            "assets/kenney/Tiles/lavaTop_low.png", "assets/kenney/Tiles/lava.png",
            "assets/kenney/Tiles/boxCrate.png", "assets/kenney/Tiles/boxCrate_double.png", "assets/kenney/Tiles/boxCrate_single.png", "assets/kenney/Tiles/boxCrate_warning.png",
            "assets/kenney/Enemies/slimeBlock.png", "assets/kenney/Enemies/slimeBlock_move.png",
            "assets/kenney/Enemies/slimePurple.png", "assets/kenney/Enemies/slimePurple_move.png",
            "assets/kenney/Enemies/slimeBlue.png", "assets/kenney/Enemies/slimeBlue_move.png",
            "assets/kenney/Enemies/slimeGreen.png", "assets/kenney/Enemies/slimeGreen_move.png",
            "assets/kenney/Enemies/mouse.png", "assets/kenney/Enemies/mouse_move.png",
            "assets/kenney/Enemies/snail.png", "assets/kenney/Enemies/snail_move.png",
            "assets/kenney/Enemies/ladybug.png", "assets/kenney/Enemies/ladybug_move.png",
            "assets/kenney/Enemies/wormGreen.png", "assets/kenney/Enemies/wormGreen_move.png",
            "assets/kenney/Enemies/wormPink.png", "assets/kenney/Enemies/wormPink_move.png",
            "assets/kenney/Enemies/sawHalf.png", "assets/kenney/Enemies/sawHalf_move.png",
            "assets/kenney/Items/coinGold.png",
            "assets/kenney/Players/128x256/Beige/alienBeige_stand.png", "assets/kenney/Players/128x256/Beige/alienBeige_jump.png",
            "assets/kenney/Players/128x256/Beige/alienBeige_walk1.png", "assets/kenney/Players/128x256/Beige/alienBeige_walk2.png",
            "assets/kenney/Players/128x256/Blue/alienBlue_stand.png", "assets/kenney/Players/128x256/Blue/alienBlue_jump.png",
            "assets/kenney/Players/128x256/Blue/alienBlue_walk1.png", "assets/kenney/Players/128x256/Blue/alienBlue_walk2.png",
            "assets/kenney/Players/128x256/Green/alienGreen_stand.png", "assets/kenney/Players/128x256/Green/alienGreen_jump.png",
            "assets/kenney/Players/128x256/Green/alienGreen_walk1.png", "assets/kenney/Players/128x256/Green/alienGreen_walk2.png",
            "assets/kenney/Players/128x256/Pink/alienPink_stand.png", "assets/kenney/Players/128x256/Pink/alienPink_jump.png",
            "assets/kenney/Players/128x256/Pink/alienPink_walk1.png", "assets/kenney/Players/128x256/Pink/alienPink_walk2.png",
            "assets/kenney/Players/128x256/Yellow/alienYellow_stand.png", "assets/kenney/Players/128x256/Yellow/alienYellow_jump.png",
            "assets/kenney/Players/128x256/Yellow/alienYellow_walk1.png", "assets/kenney/Players/128x256/Yellow/alienYellow_walk2.png",
            "assets/misc_assets/iconCircle_white.png",
            PG2_PLATFORM_BACKGROUNDS
        };
        *count = NUM_TEX;
        return names;
    }

    // System_Tilemap::get (tilemap.h:79-84): out of bounds is wall_mid. (x, y) in map space.
    static PG2_DEV int get(const uint8_t* tiles, int x, int y) {
        if (x < 0 || y < 0 || x >= W || y >= H) return WALL_MID;
        return tiles[y + x * H] & 15;
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV_NOINLINE bool step(const State& s, const CommonState& c, int env, int action, float* reward, const StepCtx& ctx) {
        const int N = s.N;
        const uint8_t* tiles = s.tiles + (size_t)env * (W * H);
        const float dt = 1.0f / SUB_STEPS;
        const int nents = s.num_ents[env];
        auto tile_at = [&](int x, int y) { return get(tiles, x, H - 1 - y); };

        // agent registers
        float ax = s.ax[env], ay = s.ay[env], avx = s.avx[env], avy = s.avy[env], agent_t = s.agent_t[env];
        bool on_ground = s.on_ground[env] != 0, face_forward = s.face_forward[env] != 0;
        float cam_x = c.cam_x[env], cam_y = c.cam_y[env];

        const float max_jump = 1.55f, gravity = 0.2f, max_speed = 0.5f, mix = 0.2f, air_control = 0.15f;
        const float movement_x = (float)((action == 6 || action == 7 || action == 8) - (action == 0 || action == 1 || action == 2));
        const bool jump = (action == 2 || action == 5 || action == 8);
        const bool fallthrough = (action == 0 || action == 3 || action == 6);

        bool alive = true, achieved_goal = false;
        for (int ss = 0; ss < SUB_STEPS; ss++) {
            // ---- System_Mob_AI::update (one mob per lane: mobs only read the tile map and their own state)
            for (int e = ctx.lane; e < nents; e += ctx.nlanes) {
                if (s.ent_type[e * N + env] != E_MOB) continue;
                float x = s.ent_x[e * N + env], y = s.ent_y[e * N + env], vx = s.ent_vx[e * N + env];
                x = __fadd_rn(x, __fmul_rn(vx, dt));
                Rect wall_sensor{ __fsub_rn(x, 0.5f), __fsub_rn(y, 0.6f), 1.0f, 0.5f };
                Rect floor_sensor{ __fsub_rn(x, 0.5f), __fadd_rn(y, 0.6f), 1.0f, 0.5f };
                CollisionResult wc = tile_collision(wall_sensor, tile_at, [](int id) { return (id == WALL_MID || id == WALL_TOP) ? COLL_FULL : COLL_NONE; });
                CollisionResult fc = tile_collision(floor_sensor, tile_at, [](int id) { return id == EMPTY ? COLL_FULL : COLL_NONE; });
                float new_x = __fadd_rn(wc.x, 0.5f);
                if (fc.collided) new_x = __fadd_rn(fc.x, 0.5f);
                x = new_x;
                if (wc.collided || fc.collided) vx = __fmul_rn(vx, -1.0f);
                s.ent_x[e * N + env] = x;
                s.ent_vx[e * N + env] = vx;
                s.ent_flip[e * N + env] = vx > 0.0f;
            }
            ctx.sync();   // the agent reads every entity's position

            // ---- System_Agent::update
            alive = true; achieved_goal = false;
            {
                float mix_x = on_ground ? mix : __fmul_rn(mix, air_control);
                avx = __fadd_rn(avx, __fmul_rn(__fmul_rn(mix_x, __fsub_rn(__fmul_rn(max_speed, movement_x), avx)), dt));
                if (fabsf(avx) < __fmul_rn(__fmul_rn(mix_x, max_speed), dt)) avx = 0.0f;
                if (jump && on_ground) avy = -max_jump;
                avy = __fadd_rn(avy, __fmul_rn(gravity, dt));
                if (fabsf(avy) > max_jump) avy = __fmul_rn(avy > 0.0f ? 1.0f : -1.0f, max_jump);
                ax = __fadd_rn(ax, __fmul_rn(avx, dt));
                ay = __fadd_rn(ay, __fmul_rn(avy, dt));
                // bounds { -0.5, -1.0, 1.0, 1.0 }
                Rect world{ __fadd_rn(ax, -0.5f), __fadd_rn(ay, -1.0f), 1.0f, 1.0f };
                CollisionResult cd = tile_collision(world, tile_at,
                    [](int id) { return (id == WALL_MID || id == WALL_TOP) ? COLL_FULL : (id == CRATE ? COLL_DOWN_ONLY : COLL_NONE); },
                    fallthrough, __fmul_rn(avy, dt), &ctx);
                float dpx = __fsub_rn(cd.x, world.x), dpy = __fsub_rn(cd.y, world.y);
                on_ground = dpy < 0.0f && cd.collided;
                ax = __fsub_rn(cd.x, -0.5f);
                ay = __fsub_rn(cd.y, -1.0f);
                world.x = __fadd_rn(ax, -0.5f);
                world.y = __fadd_rn(ay, -1.0f);
                if (dpx != 0.0f) avx = 0.0f;
                if (on_ground) avy = 0.0f;

                // hazards (saws: bounds {-0.5,-0.5,1,1}; mobs: {-0.5,-0.48,1,0.98}) and goals
                bool hit = false, got = false;
                for (int e = ctx.lane; e < nents; e += ctx.nlanes) {
                    int type = s.ent_type[e * N + env];
                    float ex = s.ent_x[e * N + env], ey = s.ent_y[e * N + env];
                    if (type == E_SAW) {
                        Rect hz{ __fadd_rn(ex, -0.5f), __fadd_rn(ey, -0.5f), 1.0f, 1.0f };
                        if (check_collision(world, hz)) hit = true;
                    } else if (type == E_MOB) {
                        Rect hz{ __fadd_rn(ex, -0.5f), __fadd_rn(ey, -0.48f), 1.0f, 0.98f };
                        if (check_collision(world, hz)) hit = true;
                    } else if (type == E_COIN) {
                        Rect gl{ __fadd_rn(ex, -0.5f), __fadd_rn(ey, -0.5f), 1.0f, 1.0f };
                        if (check_collision(world, gl)) got = true;
                    }
                }
                if (ctx.any(hit)) alive = false;
                if (ctx.any(got)) achieved_goal = true;
                CollisionResult lava = tile_collision(world, tile_at, [](int id) { return (id == LAVA_MID || id == LAVA_TOP) ? COLL_FULL : COLL_NONE; },
                                                      false, 0.0f, &ctx);
                if (lava.collided) alive = false;

                cam_x = __fmul_rn(ax, UNIT_TO_PIXELS);
                cam_y = __fmul_rn(__fsub_rn(ay, 0.5f), UNIT_TO_PIXELS);
                agent_t = __fadd_rn(agent_t, __fmul_rn(0.1f, dt));
                agent_t = fmodf(agent_t, 1.0f);
                if (movement_x > 0.0f) face_forward = true;
                else if (movement_x < 0.0f) face_forward = false;
            }

            // ---- System_Particles::update + System_Sprite_Render::update (animation), one entity per lane.
            // Every load of the entity is issued before the first store (stores cannot be proven not to alias later loads).
            for (int e = ctx.lane; e < nents; e += ctx.nlanes) {
                const int type = s.ent_type[e * N + env];
                const bool mob = type == E_MOB, animated = type == E_MOB || type == E_SAW;
                float life[NPART];
#pragma unroll
                for (int i = 0; i < NPART; i++) life[i] = mob ? s.part_life[(e * NPART + i) * N + env] : 1.0f;
                float timer = mob ? s.part_timer[e * N + env] : 0.0f;
                const float ent_x = mob ? s.ent_x[e * N + env] : 0.0f, ent_y = mob ? s.ent_y[e * N + env] : 0.0f;
                float anim_t = animated ? s.ent_anim_t[e * N + env] : 0.0f;
                const int frame = animated ? s.ent_frame[e * N + env] : 0;
                if (mob) {
                    int dead_index = -1;
#pragma unroll
                    for (int i = 0; i < NPART; i++) {
                        life[i] = __fsub_rn(life[i], dt);
                        if (life[i] <= 0.0f) dead_index = i;
                    }
#pragma unroll
                    for (int i = 0; i < NPART; i++) s.part_life[(e * NPART + i) * N + env] = life[i];
                    timer = __fadd_rn(timer, dt);
                    if (dead_index != -1 && timer >= 0.5f) {
                        timer = fmodf(timer, 0.5f);
                        int pi = (e * NPART + dead_index) * N + env;
                        s.part_life[pi] = 5.0f;
                        s.part_x[pi] = __fadd_rn(ent_x, 0.0f);
                        s.part_y[pi] = __fadd_rn(ent_y, 0.34f);
                    }
                    s.part_timer[e * N + env] = timer;
                }
                if (animated) {
                    const float rate = type == E_SAW ? 1.0f : 0.2f;
                    float t = __fadd_rn(anim_t, dt);
                    int adv = f2i(__fmul_rn(t, rate));
                    t = __fsub_rn(t, __fdiv_rn((float)adv, rate));
                    s.ent_anim_t[e * N + env] = t;
                    s.ent_frame[e * N + env] = (uint8_t)((frame + adv) % 2);
                }
            }
            if (!alive || achieved_goal) break;
        }

        if (ctx.leader()) {
            s.ax[env] = ax; s.ay[env] = ay; s.avx[env] = avx; s.avy[env] = avy; s.agent_t[env] = agent_t;
            s.on_ground[env] = on_ground; s.face_forward[env] = face_forward;
            c.cam_x[env] = cam_x; c.cam_y[env] = cam_y;
            c.sprites_valid[env] = 1;
        }
        *reward = achieved_goal ? 10.0f : 0.0f;      // result.second * 10.0f
        return !alive || achieved_goal;
    }

    // ---------------------------------------------------------------------------------------
    struct Gen {   // level-generation scratch view
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
        // staged entity records (all lanes keep identical copies in shared memory)
        uint8_t* etype = w.alloc<uint8_t>(MAX_ENTS);
        uint8_t* ekind = w.alloc<uint8_t>(MAX_ENTS);
        float* ex = w.alloc<float>(MAX_ENTS);
        float* ey = w.alloc<float>(MAX_ENTS);
        float* evx = w.alloc<float>(MAX_ENTS);
        int nents = 0;
        bool overflow = false;
        Gen g{ tiles, &w };

        // crate_type_indices is resized, never cleared (tilemap.cpp:108), but an entry is only ever
        // read for a crate tile, which always (re)writes it (tilemap.cpp:271-272): no stale state.
        w.fill<uint8_t>(tiles, W * H, 0);   // std::fill(tile_ids, empty)

        g.set_area(0, 0, W, 1, WALL_TOP);
        g.set_area(0, 0, 1, H, WALL_MID);
        g.set_area(W - 1, 0, 1, H, WALL_MID);
        g.set_area(0, H - 1, W, 1, WALL_MID);

        auto spawn = [&](int type, int x, int y, int kind, float vx) {
            if (nents >= MAX_ENTS) { overflow = true; return; }
            etype[nents] = (uint8_t)type; ekind[nents] = (uint8_t)kind;
            ex[nents] = __fadd_rn((float)x, 0.5f);
            ey[nents] = __fadd_rn((float)(H - 1 - y), 0.5f);
            evx[nents] = vx;
            nents++;
        };
        auto spawn_enemy_mob = [&](int x, int y) {   // tilemap.cpp:70-95: enemy index, then direction
            int enemy_index = w.rng.uniform_int(0, 8);
            float r = w.rng.uniform_real(0.0f, 1.0f);
            float vx = __fmul_rn(0.15f, __fsub_rn(__fmul_rn((float)(r < 0.5f), 2.0f), 1.0f));
            spawn(E_MOB, x, y, enemy_index, vx);
        };

        const float max_jump = 1.5f, gravity = 0.2f, max_speed = 0.5f;
        int difficulty = w.rng.uniform_int(1, 3);
        int num_sections = w.rng.uniform_int(difficulty, 2 * difficulty - 1);
        int curr_x = 5, curr_y = 1;
        int pit_thresh = difficulty;
        int danger_type = w.rng.uniform_int(0, 2);
        float max_dxf = __fdiv_rn(__fmul_rn(__fmul_rn(max_speed, 2.0f), max_jump), gravity);
        float max_dyf = __fdiv_rn(__fmul_rn(max_jump, max_jump), __fmul_rn(2.0f, gravity));
        int max_dx = f2i(__fsub_rn(max_dxf, 0.5f));
        int max_dy = f2i(__fsub_rn(max_dyf, 0.5f));

        for (int section = 0; section < num_sections; section++) {
            if (curr_x + 15 >= W) break;
            int difficult_offset = difficulty / 3;
            int dy = w.rng.uniform_int(1 + difficult_offset, 4 + difficult_offset);
            dy = min(dy, max_dy);
            if (curr_y >= 20 || (curr_y >= 5 && w.rng.uniform_real(0.0f, 1.0f) < 0.5f)) dy *= -1;
            int dx = w.rng.uniform_int(3 + difficult_offset, 2 * difficulty + 2 + difficult_offset);
            curr_y = max(1, curr_y + dy);
            bool use_pit = (dx > 7) && (curr_y > 3) && (w.rng.uniform_int(0, 19) >= pit_thresh);
            if (use_pit) {
                int x1 = w.rng.uniform_int(1, 3);
                int x2 = w.rng.uniform_int(1, 3);
                int pit_width = dx - x1 - x2;
                if (pit_width > max_dx) { pit_width = max_dx; x2 = dx - x1 - pit_width; }
                g.set_area_with_top(curr_x, 0, x1, curr_y, WALL_MID, WALL_TOP);
                g.set_area_with_top(curr_x + dx - x2, 0, x2, curr_y, WALL_MID, WALL_TOP);
                int lava_height = w.rng.uniform_int(1, curr_y - 3);
                switch (danger_type) {
                case 0: g.set_area_with_top(curr_x + x1, 1, pit_width, lava_height, LAVA_MID, LAVA_TOP); break;
                case 1: for (int i = 0; i < pit_width; i++) spawn(E_SAW, curr_x + x1 + i, 1, 0, 0.0f); break;
                case 2: for (int i = 0; i < pit_width; i++) spawn_enemy_mob(curr_x + x1 + i, 1); break;
                }
                if (pit_width > 4) {
                    int x3, w1;
                    if (pit_width == 5) { x3 = w.rng.uniform_int(1, 2); w1 = w.rng.uniform_int(1, 2); }
                    else if (pit_width == 6) { x3 = w.rng.uniform_int(1, 2) + 1; w1 = w.rng.uniform_int(1, 2); }
                    else { x3 = w.rng.uniform_int(1, 2) + 1; int x4 = w.rng.uniform_int(1, 2) + 1; w1 = pit_width - x3 - x4; }
                    g.set_area_with_top(curr_x + x1 + x3, curr_y - 1, w1, 1, WALL_MID, WALL_TOP);
                }
            } else {
                g.set_area_with_top(curr_x, 0, dx, curr_y, WALL_MID, WALL_TOP);
                int ob1_x = -1, ob2_x = -1;
                if (w.rng.uniform_int(0, 9) < (2 * difficulty) && dx > 3) {
                    ob1_x = curr_x + w.rng.uniform_int(1, dx - 2);
                    spawn(E_SAW, ob1_x, curr_y, 0, 0.0f);
                }
                if (w.rng.uniform_int(0, 9) < difficulty && dx > 3 && max_dx >= 4) {
                    ob1_x = curr_x + w.rng.uniform_int(1, dx - 2);
                    spawn_enemy_mob(ob1_x, curr_y);
                }
                for (int i = 0; i < 2; i++) {
                    int crate_x = curr_x + w.rng.uniform_int(1, dx - 2);
                    if (w.rng.uniform_real(0.0f, 1.0f) < 0.5f && ob1_x != crate_x && ob2_x != crate_x) {
                        int pile_height = w.rng.uniform_int(1, 3);
                        for (int j = 0; j < pile_height; j++) {
                            int ct = w.rng.uniform_int(0, 3);
                            __syncwarp();
                            // set() ignores out-of-range cells, the crate-type write does not check
                            // (tilemap.cpp:271-272); curr_y + j < 64 always holds here
                            g.set(crate_x, curr_y + j, CRATE | (ct << 4));
                            __syncwarp();
                        }
                    }
                }
            }
            curr_x += dx;
        }
        // coin
        spawn(E_COIN, curr_x, curr_y, 0, 0.0f);
        g.set_area_with_top(curr_x, 0, 1, curr_y, WALL_MID, WALL_TOP);
        g.set_area(curr_x + 1, 0, W - curr_x, H, WALL_MID);

        // ---- reset() tail (coinrun.cpp:478-503)
        int bg_index = w.rng.uniform_int(0, PG2_NUM_PLATFORM_BACKGROUNDS - 1);
        float bg_offset = w.rng.uniform_real(0.0f, 1.0f);
        int agent_theme = w.rng.uniform_int(0, 4);
        int map_theme = w.rng.uniform_int(0, 5);

        // ---- iteration orders of the ECS sets that are observable (Q4): sprite_render holds every
        // entity created above (ids 0..nents-1 inserted ascending), particles holds the mobs.
        USet<MAX_ENTS, 64>* us = w.alloc<USet<MAX_ENTS, 64>>(1);
        uint8_t* order = w.alloc<uint8_t>(MAX_ENTS);
        __syncwarp();
        us->init(s.nb_sprite[env]);
        for (int e = 0; e < nents; e++) us->insert(e);
        int n_sprite = us->order(order);
        int nb_sprite = us->nb;
        __syncwarp();
        for (int k = lane; k < n_sprite; k += WARP_LANES) s.sprite_order[k * N + env] = order[k];
        __syncwarp();
        us->init(s.nb_mob[env]);
        for (int e = 0; e < nents; e++) if (etype[e] == E_MOB) us->insert(e);
        int n_mob = us->order(order);
        int nb_mob = us->nb;
        __syncwarp();
        for (int k = lane; k < n_mob; k += WARP_LANES) s.mob_order[k * N + env] = order[k];

        // ---- write back
        uint8_t* gt = s.tiles + (size_t)env * (W * H);
        for (int i = lane; i < W * H / 4; i += WARP_LANES) ((uint32_t*)gt)[i] = ((const uint32_t*)tiles)[i];
        for (int e = lane; e < nents; e += WARP_LANES) {
            s.ent_type[e * N + env] = etype[e];
            s.ent_kind[e * N + env] = ekind[e];
            s.ent_x[e * N + env] = ex[e];
            s.ent_y[e * N + env] = ey[e];
            s.ent_vx[e * N + env] = evx[e];
            s.ent_anim_t[e * N + env] = 0.0f;
            s.ent_frame[e * N + env] = 0;
            s.ent_flip[e * N + env] = 0;
            s.part_timer[e * N + env] = 0.0f;
            for (int i = 0; i < NPART; i++) {
                int pi = (e * NPART + i) * N + env;
                s.part_x[pi] = 0.0f; s.part_y[pi] = 0.0f; s.part_life[pi] = 0.0f;
            }
        }
        if (lane == 0) {
            s.num_ents[env] = nents;
            s.num_mobs[env] = n_mob;
            s.nb_sprite[env] = nb_sprite;
            s.nb_mob[env] = nb_mob;
            s.ax[env] = 1.5f;
            s.ay[env] = __fsub_rn((float)(H - 1), 1.0f);      // tilemap->get_height() - 1 - 1.0f
            s.avx[env] = 0.0f; s.avy[env] = 0.0f;
            s.on_ground[env] = 0; s.face_forward[env] = 1; s.agent_t[env] = 0.0f;
            s.bg_index[env] = bg_index; s.bg_offset[env] = bg_offset;
            s.agent_theme[env] = agent_theme; s.map_theme[env] = map_theme;
            c.sprites_valid[env] = 0;
            if (overflow) c.fault[env] |= 1;
        }
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV int tile_class(uint32_t) { return 0; }

    template <class F>
    static PG2_DEV_NOINLINE void build_frame(const State& s, const CommonState& c, int env, F& f, const TexInfo* tex) {
        const int N = s.N;
        Camera cam{ c.cam_x[env], c.cam_y[env], __fdiv_rn(__fmul_rn(0.3f, f.view_w), 64.0f), f.view_w, f.view_h };   // game_zoom * width / obs_width
        int lx, ly, ux, uy;
        tile_window(cam, &lx, &ly, &ux, &uy);
        const int ncol = min(ux - lx + 1, MAX_WIN), nrow = min(uy - ly + 1, MAX_WIN);
        const bool sprites = c.sprites_valid[env] != 0;
        const int nents = s.num_ents[env];
        const int nmobs = sprites ? s.num_mobs[env] : 0;
        // NOTE(Q9): System_Particles::render walks the live ECS set, not the cleared draw list, so
        // particles would be drawn on the reset frame too — but every particle is dead right after
        // a reset (life = 0), so nothing is emitted either way.
        const int npart_slots = s.num_mobs[env] * NPART;
        const int nsprite = sprites ? nents : 0;
        // background (e.g. maze.cpp:402-408): the blit itself is built by build_tile_layer below
        const int bg = T_BG0 + s.bg_index[env];
        const TexInfo bt = tex[bg];
        const float bg_x = __fmul_rn(-s.bg_offset[env], __fsub_rn(__fdiv_rn((float)bt.w, (float)bt.h), 1.0f));
        const float bg_scale = __fdiv_rn(__fmul_rn(64.0f, UNIT_TO_PIXELS), (float)bt.h);
        (void)nmobs;
        // tile layer: every tile texture is 128x128
        const uint8_t* tiles = s.tiles + (size_t)env * (W * H);
        const int theme = s.map_theme[env];
        build_tile_layer(f, cam, tex, 1, lx, ly, ncol, nrow, [](int) { return (int)T_WALL_MID0; }, [&](int x, int yr) {
            const int y = H - 1 - yr;
            const int raw = (x < 0 || y < 0 || x >= W || y >= H) ? WALL_MID : tiles[y + x * H];
            const int id = raw & 15;
            return id == WALL_MID ? T_WALL_MID0 + theme : id == WALL_TOP ? T_WALL_TOP0 + theme : id == LAVA_MID ? (int)T_LAVA_MID
                 : id == LAVA_TOP ? (int)T_LAVA_TOP : id == CRATE ? T_CRATE0 + (raw >> 4) : (int)NO_TILE;
        }, bg, bg_x, 0.0f, bg_scale);
        // post blits: particles (set order x slot), sprites (std::sort order), agent
        emit_post_blits(f, tex, npart_slots + nsprite + 1, [&](int k, BlitReq& b, BlitRot&) {
            if (k < npart_slots) {
                int e = s.mob_order[(k / NPART) * N + env], i = k % NPART;
                int pi = (e * NPART + i) * N + env;
                float life = s.part_life[pi];
                if (life > 0.0f) {   // common_systems.cpp:315-337
                    float life_ratio = __fdiv_rn(__fsub_rn(5.0f, life), 5.0f);
                    float alpha = __fmul_rn(0.5f, __fsub_rn(1.0f, life_ratio));
                    float scale = __fmul_rn(0.45f, __fadd_rn(__fmul_rn(0.4f, life_ratio), 0.6f));
                    float offset_y = __fmul_rn(-life_ratio, 0.17f);
                    float pw = (float)tex[T_PARTICLE].w, ph = (float)tex[T_PARTICLE].h;
                    float px = __fsub_rn(__fmul_rn(s.part_x[pi], UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(0.5f, pw), scale));
                    float py = __fsub_rn(__fmul_rn(__fadd_rn(s.part_y[pi], offset_y), UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(0.5f, ph), scale));
                    b.plain(T_PARTICLE, px, py, cam, __fdiv_rn(__fmul_rn(scale, UNIT_TO_PIXELS), pw), alpha);
                }
            } else if (k < npart_slots + nsprite) {
                int j = k - npart_slots;
                int e = s.sprite_order[sort_perm(nsprite, j) * N + env];
                int type = s.ent_type[e * N + env];
                int t = type == E_COIN ? T_COIN : (type == E_SAW ? T_SAW0 + s.ent_frame[e * N + env]
                                                                 : T_ENEMY0 + 2 * s.ent_kind[e * N + env] + s.ent_frame[e * N + env]);
                float px = __fmul_rn(__fadd_rn(s.ent_x[e * N + env], -0.5f), UNIT_TO_PIXELS);
                float py = __fmul_rn(__fadd_rn(s.ent_y[e * N + env], -0.5f), UNIT_TO_PIXELS);
                float sc = __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, 1.0f), UNIT_TO_PIXELS), (float)tex[t].w);
                b.plain(t, px, py, cam, sc, 1.0f, s.ent_flip[e * N + env] != 0);
            } else {
                // agent (common_systems.cpp:254-278)
                float avx = s.avx[env];
                bool on_ground = s.on_ground[env] != 0;
                int pose = (fabsf(avx) < 0.01f && on_ground) ? 0 : (!on_ground ? 1 : (s.agent_t[env] > 0.5f ? 3 : 2));
                int t = T_AGENT0 + 4 * s.agent_theme[env] + pose;
                float px = __fmul_rn(__fsub_rn(s.ax[env], 0.5f), UNIT_TO_PIXELS);
                float py = __fmul_rn(__fsub_rn(s.ay[env], 2.0f), UNIT_TO_PIXELS);
                b.plain(t, px, py, cam, __fdiv_rn(UNIT_TO_PIXELS, (float)tex[t].w), 1.0f, s.face_forward[env] == 0);
            }
        });
    }
};

}  // namespace pg2
