// CaveFlyer — device restatement of /root/reference/games/caveflyer/:
//   step logic  cenv_step caveflyer.cpp:301-345; System_Agent::update common_systems.cpp:90-289;
//               System_Mob_AI::update :50-75; System_Particles::update :333-372;
//               System_Tilemap::get_collision tilemap.cpp:305-366
//   level gen   System_Tilemap::regenerate tilemap.cpp:118-278 (spawn helpers :35-116), Room_Generator
//               room_generator.cpp, reset() caveflyer.cpp:442-462
//   frame       render_game caveflyer.cpp:413-440; tilemap.cpp:280-303; common_systems.cpp:26-48, 291-326, 374-398
// hard_mode (compile-time default): 40 x 40 world; easy_mode (20 x 20) and memory_mode (45 x 45, unpruned caves) are the CaveFlyerT<0> / CaveFlyerT<2> instantiations. Entity ids per episode (SURVEY App. B): 0 goal, 1 agent,
// 2.. objects (obstacles, then targets, then enemies). The four post-prune automaton passes never feed back
// into the tile map (SURVEY Q18) and are skipped.
#pragma once
#include <type_traits>
#include "../pg2_common.cuh"
#include "../pg2_libm.cuh"
#include "../pg2_render.cuh"
#include "../pg2_roomgen.cuh"
#include "../pg2_state.cuh"
#include "../pg2_tilecoll.cuh"
#include "../pg2_uset.cuh"
#include "../pg2_warp.cuh"

namespace pg2 {

#define PG2_CAVEFLYER_FIELDS_(F, NT)                                                                \
    PG2_ENV_MAJOR(F)(uint8_t, tiles, NT) /* [y + x*H]: 0 empty, 1 wall */                          \
    F(int32_t, num_obj, 1)                                                                         \
    F(uint8_t, obj_type, 64)    /* slot-major; 1 obstacle, 2 target, 3 enemy, 0 destroyed */       \
    F(float, obj_x, 64) F(float, obj_y, 64) F(float, obj_vx, 64) F(float, obj_vy, 64)              \
    F(uint8_t, hazard_order, 64) /* iteration order of System_Hazard::entities (object slots) */   \
    F(uint8_t, sprite_order, 72) /* ... of System_Sprite_Render::entities (0 = goal, k+1 = object slot k) */ \
    F(int32_t, nb_hazard, 1) F(int32_t, nb_sprite, 1)                                              \
    F(float, goal_x, 1) F(float, goal_y, 1)                                                        \
    F(float, ax, 1) F(float, ay, 1) F(float, arot, 1) F(float, avx, 1) F(float, avy, 1)            \
    F(int32_t, next_bullet, 1) F(int32_t, num_bullets, 1) F(float, bullet_timer, 1)                \
    F(float, b_x, 32) F(float, b_y, 32) F(float, b_vx, 32) F(float, b_vy, 32) F(float, b_rot, 32) F(float, b_frame, 32) \
    F(float, p_x, 10) F(float, p_y, 10) F(float, p_dx, 10) F(float, p_dy, 10) F(float, p_rot, 10) F(float, p_life, 10) \
    F(float, p_timer, 1) F(uint8_t, p_enabled, 1)                                                  \
    F(int32_t, bg_index, 1) F(float, bg_offset, 1)

#define PG2_CAVEFLYER_FIELDS(F) PG2_CAVEFLYER_FIELDS_(F, 1600)
#define PG2_CAVEFLYER_FIELDS_MEMORY(F) PG2_CAVEFLYER_FIELDS_(F, 2048)
PG2_DEFINE_STATE(CaveFlyerState, PG2_CAVEFLYER_FIELDS)
PG2_DEFINE_STATE(CaveFlyerStateMemory, PG2_CAVEFLYER_FIELDS_MEMORY)

template <int MODE>
struct CaveFlyerT {
    using State = typename std::conditional<MODE == 2, CaveFlyerStateMemory, CaveFlyerState>::type;
    static constexpr int W = MODE == 0 ? 20 : MODE == 2 ? 45 : 40, H = W;   // world_dim (tilemap.cpp:121-126: easy 20, hard 40, memory 45)
    static constexpr int TILE_STRIDE = MODE == 2 ? 2048 : 1600;   // per-env extent of State::tiles (the field's size, whatever the world size)
    static constexpr bool PRUNE = MODE != 2;                      // should_prune (tilemap.cpp:203): memory mode keeps every cave of the automaton
    static constexpr int MAX_OBJ = 64, NB = 32, NPART = 10;
    static constexpr int SUB_STEPS = 4;
    static constexpr bool LANE_AWARE = false;   // step() supports warp-per-env (ctx) but measures faster thread-per-env (r01j)
    static constexpr int STEP_LANES = 32;       // (lane-aware games only) lanes per environment in k_step
    static constexpr int MAX_POST = 112;        // capacity of the frame's post-blit list
    static constexpr bool ROTATES = true;     // some blits are rotated
    static constexpr bool SLOW_RESET = true;   // level generation is long: run it concurrently with the render of the other envs
    static constexpr int RESET_ARENA = (MODE == 2 ? 56 : 52) * 1024;   // per-warp level-generation scratch (high water measured with PG2_ARENA_TRACE)
    static constexpr bool PREFETCH_LEVELS = true;    // the RNG is only drawn inside reset(): the next level is generated one episode ahead
    static constexpr int PREFETCH_MIN_EPISODE = 0;   // level prefetch whatever max_episode_steps is
    static const char* reset_keeps() { return " cam_x cam_y "; }   // fields reset() does not write (they persist across episodes)
    static constexpr int TILE_CLASSES = 1;
    static constexpr int WIN_ROWS = 11;        // most tile rows the camera window can span (zoom-dependent; frame table sizing)
    static constexpr int BLIT_UNROLL = 1;     // post-blit patches fetched together (pg2_render.cuh draw_blit_band)
    static constexpr int RENDER_MIN_CTAS = 7;   // CTAs per SM the register allocation of k_render aims at
    static constexpr int DEFAULT_MODE = MODE;    // this instantiation's distribution mode (the reference compiles in 1 = hard; tilemap.h Config)
    static bool mode_supported(int mode) { return mode == MODE; }
    static constexpr bool HAS_TILES = true;     // the frame has a tile layer
    static constexpr bool STATIC_VIEW = false;   // the camera follows the agent: the base image changes every frame (a camera-keyed cache measured slower)
    enum Obj { O_NONE = 0, O_OBSTACLE, O_TARGET, O_ENEMY };
    enum Tex { T_WALL = 0, T_GOAL, T_TARGET, T_OBSTACLE, T_ENEMY, T_BULLET, T_SHIP, T_PARTICLE, T_EXPL0, T_BG0 = 13, NUM_BG = 13, NUM_TEX = 26 };

    static const char* const* texture_names(int* count) {
        static const char* const names[NUM_TEX] = {
            "assets/misc_assets/groundA.png", "assets/misc_assets/ufoGreen2.png", "assets/misc_assets/ufoRed2.png",
            "assets/misc_assets/meteorBrown_big1.png", "assets/misc_assets/enemyShipBlue4.png",
            "assets/misc_assets/laserBlue02.png", "assets/misc_assets/playerShip1_red.png",
            "assets/misc_assets/towerDefense_tile295.png",
            "assets/misc_assets/explosion1.png", "assets/misc_assets/explosion2.png", "assets/misc_assets/explosion3.png",
            "assets/misc_assets/explosion4.png", "assets/misc_assets/explosion5.png",
            "assets/space_backgrounds/deep_space_01.png", "assets/space_backgrounds/spacegen_01.png",
            "assets/space_backgrounds/milky_way_01.png", "assets/space_backgrounds/ez_space_lite_01.png",
            "assets/space_backgrounds/meyespace_v1_01.png", "assets/space_backgrounds/eye_nebula_01.png",
            "assets/space_backgrounds/deep_sky_01.png", "assets/space_backgrounds/space_nebula_01.png",
            "assets/space_backgrounds/Background-1.png", "assets/space_backgrounds/Background-2.png",
            "assets/space_backgrounds/Background-3.png", "assets/space_backgrounds/Background-4.png",
            "assets/space_backgrounds/parallax-space-backgound.png",
        };
        *count = NUM_TEX;
        return names;
    }

    // System_Tilemap::get (tilemap.h:79-84): out of bounds is a wall. (x, y) in map space.
    static PG2_DEV int get(const uint8_t* tiles, int x, int y) {
        if (x < 0 || y < 0 || x >= W || y >= H) return 1;
        return tiles[y + x * H];
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV_NOINLINE bool step(const State& s, const CommonState& c, int env, int action, float* reward, const StepCtx& ctx) {
        const int N = s.N;
        const uint8_t* tiles = s.tiles + (size_t)env * TILE_STRIDE;
        const float dt = 1.0f / SUB_STEPS;
        const double PI = 3.14159265358979323846;
        const int nobj = s.num_obj[env];
        auto tile_at = [&](int x, int y) { return get(tiles, x, H - 1 - y); };
        auto wall = [](int id) { return id == 1 ? COLL_FULL : COLL_NONE; };
        auto obj_rect = [&](int k) {
            float x = s.obj_x[k * N + env], y = s.obj_y[k * N + env];
            return s.obj_type[k * N + env] == O_ENEMY ? Rect{ __fadd_rn(x, -0.4f), __fadd_rn(y, -0.4f), 0.8f, 0.8f }
                                                      : Rect{ __fadd_rn(x, -0.25f), __fadd_rn(y, -0.25f), 0.5f, 0.5f };
        };

        float ax = s.ax[env], ay = s.ay[env], rot = s.arot[env], avx = s.avx[env], avy = s.avy[env];
        int next_bullet = s.next_bullet[env], num_bullets = s.num_bullets[env];
        float bullet_timer = s.bullet_timer[env];
        float p_timer = s.p_timer[env];
        bool p_enabled = s.p_enabled[env] != 0;
        float cam_x = c.cam_x[env], cam_y = c.cam_y[env];
        const Rect goal_rect{ __fadd_rn(s.goal_x[env], -0.4f), __fadd_rn(s.goal_y[env], -0.4f), 0.8f, 0.8f };

        const float movement_x = (float)((action == 6 || action == 7 || action == 8) - (action == 0 || action == 1 || action == 2));
        float movement_y = (float)((action == 2 || action == 5 || action == 8) - (action == 0 || action == 3 || action == 6));
        const bool fire = action == 9;
        if (movement_y < 0.0f) movement_y = __fmul_rn(movement_y, 0.5f);

        bool alive = true, achieved_goal = false;
        int targets_destroyed = 0;
        for (int ss = 0; ss < SUB_STEPS; ss++) {
            // ================= System_Agent::update =================
            alive = true; achieved_goal = false; targets_destroyed = 0;
            {
                rot = __fadd_rn(rot, __fmul_rn(__fmul_rn(movement_x, 0.05f), dt));
                float dir_x, dir_y;
                glibc_sincosf(rot, &dir_y, &dir_x);
                if (fire) {
                    if (bullet_timer == 0.0f && num_bullets < NB) {
                        bullet_timer = 0.5f;
                        int i = next_bullet * N + env;
                        s.b_rot[i] = rot;
                        s.b_vx[i] = __fmul_rn(dir_x, 1.0f); s.b_vy[i] = __fmul_rn(dir_y, 1.0f);
                        s.b_x[i] = ax; s.b_y[i] = ay; s.b_frame[i] = 0.0f;
                        next_bullet = (next_bullet + 1) % NB;
                        num_bullets++;
                    } else bullet_timer = fmaxf(0.0f, __fsub_rn(bullet_timer, dt));
                }
                float acc_x = __fmul_rn(__fmul_rn(dir_x, movement_y), 0.05f), acc_y = __fmul_rn(__fmul_rn(dir_y, movement_y), 0.05f);
                avx = __fadd_rn(avx, __fmul_rn(__fsub_rn(acc_x, __fmul_rn(avx, 0.1f)), dt));
                avy = __fadd_rn(avy, __fmul_rn(__fsub_rn(acc_y, __fmul_rn(avy, 0.1f)), dt));
                ax = __fadd_rn(ax, __fmul_rn(avx, dt));
                ay = __fadd_rn(ay, __fmul_rn(avy, dt));
                Rect world{ __fadd_rn(ax, -0.4f), __fadd_rn(ay, -0.4f), 0.8f, 0.8f };
                CollisionResult cd = tile_collision(world, tile_at, wall);
                float dpx = __fsub_rn(cd.x, world.x), dpy = __fsub_rn(cd.y, world.y);
                ax = __fsub_rn(cd.x, -0.4f);
                ay = __fsub_rn(cd.y, -0.4f);
                world.x = __fadd_rn(ax, -0.4f); world.y = __fadd_rn(ay, -0.4f);
                if (dpx != 0.0f) avx = 0.0f;
                if (dpy != 0.0f) avy = 0.0f;
                bool hit = false;
                for (int o = ctx.lane; o < nobj; o += ctx.nlanes)
                    if (s.obj_type[o * N + env] != O_NONE && check_collision(world, obj_rect(o))) hit = true;
                if (ctx.any(hit)) alive = false;
                if (check_collision(world, goal_rect)) achieved_goal = true;
                cam_x = __fmul_rn(ax, UNIT_TO_PIXELS);
                cam_y = __fmul_rn(ay, UNIT_TO_PIXELS);

                for (int i = 0; i < num_bullets; i++) {
                    int bi = ((NB + next_bullet - 1 - i) % NB) * N + env;
                    float frame = s.b_frame[bi];
                    if (frame == -1.0f) continue;
                    float x = s.b_x[bi], y = s.b_y[bi], vx = s.b_vx[bi], vy = s.b_vy[bi];
                    if (frame == 0.0f) {
                        Rect bw{ __fsub_rn(x, 0.01f), __fsub_rn(y, 0.01f), 0.02f, 0.02f };
                        CollisionResult bc = tile_collision(bw, tile_at, wall);
                        if (bc.collided) { vx = 0.0f; vy = 0.0f; frame = 1.0f; }
                        for (int k = 0; k < nobj; k++) {
                            int o = s.hazard_order[k * N + env];
                            int type = s.obj_type[o * N + env];
                            if (type == O_NONE) continue;
                            if (check_collision(bw, obj_rect(o))) {
                                vx = 0.0f; vy = 0.0f; frame = 1.0f;
                                if (type == O_TARGET) { s.obj_type[o * N + env] = O_NONE; targets_destroyed++; }
                                break;
                            }
                        }
                    }
                    x = __fadd_rn(x, __fmul_rn(vx, dt));
                    y = __fadd_rn(y, __fmul_rn(vy, dt));
                    if (frame >= 5.0f) { num_bullets--; frame = -1.0f; }
                    else if (frame >= 1.0f) frame = __fadd_rn(frame, __fmul_rn(0.5f, dt));
                    s.b_x[bi] = x; s.b_y[bi] = y; s.b_vx[bi] = vx; s.b_vy[bi] = vy; s.b_frame[bi] = frame;
                }
                p_enabled = movement_y > 0.0f;
            }

            // ================= System_Mob_AI::update (one enemy per lane) =================
            ctx.sync();
            for (int o = ctx.lane; o < nobj; o += ctx.nlanes) {
                if (s.obj_type[o * N + env] != O_ENEMY) continue;
                float x = s.obj_x[o * N + env], y = s.obj_y[o * N + env], vx = s.obj_vx[o * N + env], vy = s.obj_vy[o * N + env];
                x = __fadd_rn(x, __fmul_rn(vx, dt));
                y = __fadd_rn(y, __fmul_rn(vy, dt));
                Rect wc{ __fadd_rn(x, -0.4f), __fadd_rn(y, -0.4f), 0.8f, 0.8f };
                if (tile_collision(wc, tile_at, wall).collided) { vx = -vx; vy = -vy; }
                s.obj_x[o * N + env] = x; s.obj_y[o * N + env] = y; s.obj_vx[o * N + env] = vx; s.obj_vy[o * N + env] = vy;
            }

            // ================= System_Particles::update =================
            ctx.sync();
            {
                int dead_index = -1;
                float life[NPART];   // fetched before the first store: the stores cannot be proven not to alias the loads
#pragma unroll
                for (int i = 0; i < NPART; i++) life[i] = s.p_life[i * N + env];
#pragma unroll
                for (int i = 0; i < NPART; i++) {
                    life[i] = __fsub_rn(life[i], dt);
                    if (life[i] <= 0.0f) dead_index = i;
                }
#pragma unroll
                for (int i = 0; i < NPART; i++) s.p_life[i * N + env] = life[i];
                p_timer = __fadd_rn(p_timer, dt);
                if (dead_index != -1 && p_timer >= 0.3f && p_enabled) {
                    p_timer = fmodf(p_timer, 0.3f);
                    int pi = dead_index * N + env;
                    s.p_life[pi] = 3.0f;
                    float prot = (float)__dadd_rn((double)rot, __dmul_rn(PI, 0.5));
                    s.p_rot[pi] = prot;
                    float sn, cs, sr, cr;
                    glibc_sincosf(prot, &sn, &cs);
                    glibc_sincosf(rot, &sr, &cr);
                    s.p_dx[pi] = -cr; s.p_dy[pi] = -sr;
                    // offset { 0.0f, 0.3f }
                    float ox = __fsub_rn(__fmul_rn(cs, 0.0f), __fmul_rn(sn, 0.3f));
                    float oy = __fadd_rn(__fmul_rn(sn, 0.0f), __fmul_rn(cs, 0.3f));
                    s.p_x[pi] = __fadd_rn(ax, ox);
                    s.p_y[pi] = __fadd_rn(ay, oy);
                }
            }
            if (!alive || achieved_goal) break;
        }

        ctx.sync();
        if (ctx.leader()) {
            s.ax[env] = ax; s.ay[env] = ay; s.arot[env] = rot; s.avx[env] = avx; s.avy[env] = avy;
            s.next_bullet[env] = next_bullet; s.num_bullets[env] = num_bullets; s.bullet_timer[env] = bullet_timer;
            s.p_timer[env] = p_timer; s.p_enabled[env] = p_enabled;
            c.cam_x[env] = cam_x; c.cam_y[env] = cam_y;
            c.sprites_valid[env] = 1;
        }
        *reward = __fadd_rn(__fmul_rn((float)achieved_goal, 10.0f), __fmul_rn((float)targets_destroyed, 3.0f));
        return !alive || achieved_goal;
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV int check_neighbors(float p0x, float p0y, float p1x, float p1y) {   // tilemap.cpp:104-116
        if (fabsf(__fsub_rn(p0x, p1x)) <= 0.001f && fabsf(__fsub_rn(p0y, p1y)) <= 2.0f) return 1;
        if (fabsf(__fsub_rn(p0x, p1x)) <= 2.0f && fabsf(__fsub_rn(p0y, p1y)) <= 0.001f) return 2;
        return 0;
    }

    static PG2_DEV_NOINLINE void regenerate(const State& s, const CommonState& c, int env, WarpCtx& w) {
        const int N = s.N, lane = w.lane;
        RoomGen rg;
        rg.init(w, W, H);
        uint8_t* tiles = w.alloc<uint8_t>(W * H);      // 0 empty, 1 wall, 2 marker
        uint16_t* free_cells = rg.queue;               // reused once the searches are done
        uint16_t* obstacle_indices = w.alloc<uint16_t>(MAX_OBJ);
        uint8_t* otype = w.alloc<uint8_t>(MAX_OBJ);
        float* ox = w.alloc<float>(MAX_OBJ);
        float* oy = w.alloc<float>(MAX_OBJ);
        float* ovx = w.alloc<float>(MAX_OBJ);
        float* ovy = w.alloc<float>(MAX_OBJ);
        uint8_t* order = w.alloc<uint8_t>(MAX_OBJ + 8);
        USet<MAX_OBJ + 8, 128>* us = w.alloc<USet<MAX_OBJ + 8, 128>>(1);
        bool fault = false;

        w.rng.bernoulli_fill(rg.grid, W * H, [](int) { return 0.5f; });   // grid[i] = dist01(rng) < 0.5f ? 1 : 0
        rg.update(w);
        rg.update(w);
        int nroom = rg.find_best_room(w);
        if (nroom <= 0) { fault = true; nroom = 1; rg.order[0] = 0; }     // Q20: assert(!best_room.empty())

        int goal_index = w.rng.uniform_int(0, nroom - 1);
        int agent_index = w.rng.uniform_int(0, nroom - 1);
        if (agent_index == goal_index) agent_index = (agent_index + 1) % nroom;
        const int goal_cell = rg.order[goal_index], agent_cell = rg.order[agent_index];
        const float goal_x = __fadd_rn((float)(goal_cell / H), 0.5f), goal_y = __fadd_rn((float)(H - 1 - goal_cell % H), 0.5f);
        const float agent_x = __fadd_rn((float)(agent_cell / H), 0.5f), agent_y = (float)(H - 1 - (agent_cell % H));

        int plen = rg.find_path(w, agent_cell, goal_cell);
        if (PRUNE) {   // only wide_path = goal_path dilated 4 times stays open
            rg.expand(w, rg.path, plen, 4, rg.mark);
            for (int i = lane; i < W * H; i += WARP_LANES) tiles[i] = rg.mark[i] ? 0 : 1;
        } else {       // the automaton's grid as it is (tilemap.cpp:152-160; best_room's cells are spaces of it already)
            for (int i = lane; i < W * H; i += WARP_LANES) tiles[i] = rg.grid[i] == 1 ? 1 : 0;
        }
        __syncwarp();
        for (int i = lane; i < plen; i += WARP_LANES) tiles[rg.path[i]] = 2;
        __syncwarp();
        const int nfree = warp_compact(w, W * H, [&](int i) { return tiles[i] == 0; }, free_cells);

        const int chunk = nfree / 80;
        int num_objects = 3 * chunk;
        if (num_objects > MAX_OBJ) { fault = true; num_objects = MAX_OBJ; }
        for (int i = 0; i < num_objects; i++) {
            int index = w.rng.uniform_int(0, nfree - 1);
            bool repeat;
            do {
                repeat = false;
                for (int j = 0; j < i; j++)
                    if (obstacle_indices[j] == index) { index = (index + 1) % nfree; repeat = true; break; }
            } while (repeat);
            __syncwarp();
            obstacle_indices[i] = (uint16_t)index;
            int cell = free_cells[index];
            float x = __fadd_rn((float)(cell / H), 0.5f), y = __fadd_rn((float)(H - 1 - cell % H), 0.5f);
            float vx = 0.0f, vy = 0.0f;
            int type = i < chunk ? O_OBSTACLE : (i < 2 * chunk ? O_TARGET : O_ENEMY);
            if (type == O_ENEMY) {
                // magnitude is drawn before the sign (SURVEY Q15)
                float mag = __fadd_rn(__fmul_rn(0.1f, w.rng.uniform_real(0.0f, 1.0f)), 0.1f);
                float vel = __fmul_rn(mag, w.rng.uniform_real(0.0f, 1.0f) < 0.5f ? 1.0f : -1.0f);
                int coll = check_neighbors(x, y, agent_x, agent_y);
                if (coll == 0) { if (w.rng.uniform_real(0.0f, 1.0f) < 0.5f) vx = vel; else vy = vel; }
                else if (coll == 1) vx = vel;
                else vy = vel;
            }
            otype[i] = (uint8_t)type; ox[i] = x; oy[i] = y; ovx[i] = vx; ovy[i] = vy;
            __syncwarp();
        }

        // ---- reset() tail
        int bg_index = w.rng.uniform_int(0, NUM_BG - 1);
        float bg_offset = w.rng.uniform_real(0.0f, 1.0f);

        // ---- ECS set orders. hazard: objects (entity ids 2..); sprite_render: goal (id 0) + objects
        us->init(s.nb_hazard[env]);
        for (int k = 0; k < num_objects; k++) us->insert(2 + k);
        int nh = us->order(order);
        int nb_hazard = us->nb;
        __syncwarp();
        for (int k = lane; k < nh; k += WARP_LANES) s.hazard_order[k * N + env] = (uint8_t)(order[k] - 2);
        __syncwarp();
        us->init(s.nb_sprite[env]);
        us->insert(0);
        for (int k = 0; k < num_objects; k++) us->insert(2 + k);
        int nsp = us->order(order);
        int nb_sprite = us->nb;
        __syncwarp();
        for (int k = lane; k < nsp; k += WARP_LANES) s.sprite_order[k * N + env] = (uint8_t)(order[k] == 0 ? 0 : order[k] - 1);

        uint8_t* gt = s.tiles + (size_t)env * TILE_STRIDE;
        for (int i = lane; i < W * H; i += WARP_LANES) gt[i] = tiles[i] == 1 ? 1 : 0;   // markers cleared
        for (int k = lane; k < num_objects; k += WARP_LANES) {
            s.obj_type[k * N + env] = otype[k];
            s.obj_x[k * N + env] = ox[k]; s.obj_y[k * N + env] = oy[k];
            s.obj_vx[k * N + env] = ovx[k]; s.obj_vy[k * N + env] = ovy[k];
        }
        for (int k = lane; k < NB; k += WARP_LANES) s.b_frame[k * N + env] = -1.0f;
        for (int k = lane; k < NPART; k += WARP_LANES) {
            s.p_x[k * N + env] = 0.0f; s.p_y[k * N + env] = 0.0f; s.p_dx[k * N + env] = 0.0f; s.p_dy[k * N + env] = 0.0f;
            s.p_rot[k * N + env] = 0.0f; s.p_life[k * N + env] = 0.0f;
        }
        if (lane == 0) {
            s.num_obj[env] = num_objects;
            s.nb_hazard[env] = nb_hazard; s.nb_sprite[env] = nb_sprite;
            s.goal_x[env] = goal_x; s.goal_y[env] = goal_y;
            s.ax[env] = agent_x; s.ay[env] = agent_y; s.arot[env] = 0.0f; s.avx[env] = 0.0f; s.avy[env] = 0.0f;
            s.next_bullet[env] = 0; s.num_bullets[env] = 0; s.bullet_timer[env] = 0.0f;
            s.p_timer[env] = 0.0f; s.p_enabled[env] = 1;
            s.bg_index[env] = bg_index; s.bg_offset[env] = bg_offset;
            c.sprites_valid[env] = 0;
            if (fault) c.fault[env] |= 1;
        }
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV int tile_class(uint32_t) { return 0; }

    template <class F>
    static PG2_DEV_NOINLINE void build_frame(const State& s, const CommonState& c, int env, F& f, const TexInfo* tex) {
        const int N = s.N;
        const double PI = 3.14159265358979323846;
        Camera cam{ c.cam_x[env], c.cam_y[env], __fdiv_rn(__fmul_rn(0.5f, f.view_w), 64.0f), f.view_w, f.view_h };
        int lx, ly, ux, uy;
        tile_window(cam, &lx, &ly, &ux, &uy);
        const int ncol = min(ux - lx + 1, MAX_WIN), nrow = min(uy - ly + 1, MAX_WIN);
        const int nobj = s.num_obj[env];
        const bool sprites = c.sprites_valid[env] != 0;
        // background (e.g. maze.cpp:402-408): the blit itself is built by build_tile_layer below
        const int bg = T_BG0 + s.bg_index[env];
        const TexInfo bt = tex[bg];
        const float bg_x = __fmul_rn(-s.bg_offset[env], __fsub_rn(__fdiv_rn((float)bt.w, (float)bt.h), 1.0f));
        const float bg_scale = __fdiv_rn(__fmul_rn(64.0f, UNIT_TO_PIXELS), (float)bt.h);
        auto sprite_alive = [&](int sp) { return sp == 0 || s.obj_type[(sp - 1) * N + env] != O_NONE; };
        const int nlive = live_list(f, sprites ? nobj + 1 : 0, [&](int j) {
            const int sp = s.sprite_order[j * N + env];
            return sprite_alive(sp) ? sp : -1; });
        const int num_bullets = s.num_bullets[env], next_bullet = s.next_bullet[env];
        const int o_spr = NPART, o_bul = o_spr + nlive, o_ship = o_bul + num_bullets;
        const uint8_t* tiles = s.tiles + (size_t)env * TILE_STRIDE;
        build_tile_layer(f, cam, tex, 1, lx, ly, ncol, nrow, [](int) { return (int)T_WALL; },
                         [&](int x, int y) { return get(tiles, x, H - 1 - y) == 1 ? (int)T_WALL : (int)NO_TILE; }, bg, bg_x, 0.0f, bg_scale);
        emit_post_blits(f, tex, o_ship + 1, [&](int k, BlitReq& b, BlitRot& rot) {
            if (k < o_spr) {   // System_Particles::render
                int pi = k * N + env;
                float life = s.p_life[pi];
                if (life <= 0.0f) return;
                float life_ratio = __fdiv_rn(__fsub_rn(3.0f, life), 3.0f);
                float alpha = __fmul_rn(0.5f, __fsub_rn(1.0f, life_ratio));
                float scale = __fmul_rn(1.0f, __fadd_rn(__fmul_rn(0.4f, life_ratio), 0.6f));
                float shift = __fmul_rn(life_ratio, 2.0f);
                float pw = (float)tex[T_PARTICLE].w, ph = (float)tex[T_PARTICLE].h;
                float size = __fdiv_rn(__fmul_rn(scale, UNIT_TO_PIXELS), pw);
                float x = __fsub_rn(__fmul_rn(__fadd_rn(s.p_x[pi], __fmul_rn(s.p_dx[pi], shift)), UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(size, pw), 0.5f));
                float y = __fsub_rn(__fmul_rn(__fadd_rn(s.p_y[pi], __fmul_rn(s.p_dy[pi], shift)), UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(size, ph), 0.5f));
                b.rotated(T_PARTICLE, x, y, cam, s.p_rot[pi], size, alpha, &rot);
            } else if (k < o_bul) {
                const int sp = f.live[sort_perm(nlive, k - o_spr)];
                int t; float x, y;
                if (sp == 0) { t = T_GOAL; x = s.goal_x[env]; y = s.goal_y[env]; }
                else {
                    int o = sp - 1, type = s.obj_type[o * N + env];
                    t = type == O_OBSTACLE ? T_OBSTACLE : (type == O_TARGET ? T_TARGET : T_ENEMY);
                    x = s.obj_x[o * N + env]; y = s.obj_y[o * N + env];
                }
                float px = __fmul_rn(__fadd_rn(x, -0.4f), UNIT_TO_PIXELS);
                float py = __fmul_rn(__fadd_rn(y, -0.4f), UNIT_TO_PIXELS);
                float sc = __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, 0.8f), UNIT_TO_PIXELS), (float)tex[t].w);
                b.plain(t, px, py, cam, sc);
            } else if (k < o_ship) {
                int bi = ((NB + next_bullet - 1 - (k - o_bul)) % NB) * N + env;
                float frame = s.b_frame[bi];
                if (frame == -1.0f) return;
                int t = frame == 0.0f ? T_BULLET : T_EXPL0 + f2i(__fsub_rn(frame, 1.0f));
                const float size = 0.1f;
                float x = __fsub_rn(__fmul_rn(s.b_x[bi], UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(size, (float)tex[t].w), 0.5f));
                float y = __fsub_rn(__fmul_rn(s.b_y[bi], UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(size, (float)tex[t].h), 0.5f));
                float rotation = (float)__dadd_rn((double)s.b_rot[bi], __dmul_rn(PI, 0.5));
                b.rotated(t, x, y, cam, rotation, size, 1.0f, &rot);
            } else {
                const float size = 0.15f;
                float x = __fsub_rn(__fmul_rn(s.ax[env], UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(size, (float)tex[T_SHIP].w), 0.5f));
                float y = __fsub_rn(__fmul_rn(s.ay[env], UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(size, (float)tex[T_SHIP].h), 0.5f));
                float rotation = (float)__dadd_rn((double)s.arot[env], __dmul_rn(PI, 0.5));
                b.rotated(T_SHIP, x, y, cam, rotation, size, 1.0f, &rot);
            }
        });
    }
};
using CaveFlyer = CaveFlyerT<1>;

}  // namespace pg2
