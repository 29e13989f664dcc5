// Jumper — device restatement of /root/reference/games/jumper/:
//   step logic  cenv_step jumper.cpp:340-385; System_Agent::update common_systems.cpp:57-202;
//               System_Particles::update :250-279; System_Tilemap::get_collision tilemap.cpp:280-341
//   level gen   System_Tilemap::regenerate tilemap.cpp:79-253 (helpers :41-77), Maze_Generator
//               maze_generator.cpp:47-173, Room_Generator room_generator.cpp, reset() jumper.cpp:512-535
//   frame       render_game incl. compass HUD jumper.cpp:445-510; tilemap.cpp:255-278;
//               common_systems.cpp:26-48, 204-244, 281-303
// hard_mode (compile-time default): 40 x 40 world; easy_mode (20 x 20) and memory_mode (45 x 45, unpruned cave, no spikes) are the JumperT<0> / JumperT<2> instantiations. Entity ids (SURVEY App. B): 0 goal, 1 agent, 2.. spikes.
#pragma once
#include <type_traits>
#include "../pg2_common.cuh"
#include "../pg2_libm.cuh"
#include "../pg2_mazegen.cuh"
#include "../pg2_render.cuh"
#include "../pg2_roomgen.cuh"
#include "../pg2_state.cuh"
#include "../pg2_tilecoll.cuh"
#include "../pg2_uset.cuh"
#include "../pg2_warp.cuh"
#include "platform_bgs.h"

namespace pg2 {

#define PG2_JUMPER_FIELDS_(F, NT)                                                                   \
    PG2_ENV_MAJOR(F)(uint8_t, tiles, NT) /* [y + x*H]: 0 empty, 1 wall_top, 2 wall_mid */          \
    F(int32_t, num_spikes, 1)                                                                      \
    F(uint16_t, spike_cell, 64) /* slot-major */                                                   \
    F(uint8_t, sprite_order, 72) /* iteration order of System_Sprite_Render::entities: 0 goal, k+1 spike k */ \
    F(int32_t, nb_sprite, 1)                                                                       \
    F(float, goal_x, 1) F(float, goal_y, 1)                                                        \
    F(float, ax, 1) F(float, ay, 1) F(float, avx, 1) F(float, avy, 1)                              \
    F(uint8_t, on_ground, 1) F(uint8_t, face_forward, 1) F(float, agent_t, 1)                      \
    F(float, jump_timer, 1) F(int32_t, jumps_left, 1)                                              \
    F(float, to_goal_x, 1) F(float, to_goal_y, 1)   /* System_Agent::info.to_goal: survives reset() (App. A) */ \
    F(float, p_x, 10) F(float, p_y, 10) F(float, p_life, 10) F(float, p_timer, 1) F(uint8_t, p_enabled, 1) \
    F(int32_t, bg_index, 1) F(float, bg_offset, 1) F(int32_t, map_theme, 1)

#define PG2_JUMPER_FIELDS(F) PG2_JUMPER_FIELDS_(F, 1600)
#define PG2_JUMPER_FIELDS_MEMORY(F) PG2_JUMPER_FIELDS_(F, 2048)
PG2_DEFINE_STATE(JumperState, PG2_JUMPER_FIELDS)
PG2_DEFINE_STATE(JumperStateMemory, PG2_JUMPER_FIELDS_MEMORY)

template <int MODE>
struct JumperT {
    using State = typename std::conditional<MODE == 2, JumperStateMemory, JumperState>::type;
    static constexpr int W = MODE == 0 ? 20 : MODE == 2 ? 45 : 40, H = W;   // world_dim (tilemap.cpp:82-87: easy 20, hard 40, memory 45)
    static constexpr int TILE_STRIDE = MODE == 2 ? 2048 : 1600;   // per-env extent of State::tiles (the field's size, whatever the world size)
    static constexpr bool PRUNE = MODE != 2;                      // should_prune (tilemap.cpp:176): memory mode keeps the whole cave
    static constexpr float SPIKE_PROB = MODE == 2 ? 0.0f : 0.2f;  // tilemap.cpp:205 (the draw happens either way)
    static constexpr int MAX_SPIKES = 64, NPART = 10;
    static constexpr int SUB_STEPS = 4;
    static constexpr bool LANE_AWARE = false;   // step() supports warp-per-env (ctx) but measures faster thread-per-env (r01j)
    static constexpr int STEP_LANES = 32;       // (lane-aware games only) lanes per environment in k_step
    static constexpr int MAX_POST = 80;        // capacity of the frame's post-blit list
    static constexpr bool ROTATES = true;     // some blits are rotated
    static constexpr bool SLOW_RESET = true;   // level generation is long: run it concurrently with the render of the other envs
    static constexpr int RESET_ARENA = (MODE == 2 ? 64 : 52) * 1024;   // per-warp level-generation scratch (high water measured with PG2_ARENA_TRACE)
    static constexpr bool PREFETCH_LEVELS = true;    // the RNG is only drawn inside reset(): the next level is generated one episode ahead
    static constexpr int PREFETCH_MIN_EPISODE = 0;   // level prefetch whatever max_episode_steps is
    static const char* reset_keeps() { return " cam_x cam_y to_goal_x to_goal_y "; }   // fields reset() does not write (they persist across episodes)
    static constexpr int TILE_CLASSES = 2;
    static constexpr int WIN_ROWS = 16;        // most tile rows the camera window can span (zoom-dependent; frame table sizing)
    static constexpr int BLIT_UNROLL = 1;     // post-blit patches fetched together (pg2_render.cuh draw_blit_band)
    static constexpr int RENDER_MIN_CTAS = 7;   // CTAs per SM the register allocation of k_render aims at
    static constexpr int DEFAULT_MODE = MODE;    // this instantiation's distribution mode (the reference compiles in 1 = hard; tilemap.h Config)
    static bool mode_supported(int mode) { return mode == MODE; }
    static constexpr bool HAS_TILES = true;     // the frame has a tile layer
    static constexpr bool STATIC_VIEW = false;   // the camera follows the agent: the base image changes every frame (a camera-keyed cache measured slower)
    enum Tile { EMPTY = 0, WALL_TOP, WALL_MID, SPIKE };
    enum Tex {
        T_WALL_TOP0 = 0, T_WALL_MID0 = 4, T_SPIKE = 8, T_CARROT, T_STAND, T_JUMP, T_WALK1, T_WALK2, T_PARTICLE,
        T_CIRCLE, T_NEEDLE, T_BAR, T_BG0 = 18, NUM_TEX = 18 + PG2_NUM_PLATFORM_BACKGROUNDS
    };

    static const char* const* texture_names(int* count) {
        static const char* const names[NUM_TEX] = {
            "assets/platformer/tileBlue_05.png", "assets/platformer/tileGreen_05.png",
            "assets/platformer/tileYellow_06.png", "assets/platformer/tileBrown_06.png",
            "assets/platformer/tileBlue_08.png", "assets/platformer/tileGreen_08.png",
            "assets/platformer/tileYellow_09.png", "assets/platformer/tileBrown_09.png",
            "assets/misc_assets/spikeMan_stand.png", "assets/misc_assets/carrot.png",
            "assets/misc_assets/bunny2_ready.png", "assets/misc_assets/bunny2_jump.png",
            "assets/misc_assets/bunny2_walk1.png", "assets/misc_assets/bunny2_walk2.png",
            "assets/misc_assets/iconCircle_white.png",
            "assets/custom/jumper_compass_circle.png", "assets/custom/jumper_compass_needle.png", "assets/custom/jumper_compass_bar.png",
            PG2_PLATFORM_BACKGROUNDS
        };
        *count = NUM_TEX;
        return names;
    }

    // System_Tilemap::get (tilemap.h:83-88): out of bounds is wall_mid. (x, y) in map space.
    static PG2_DEV int get(const uint8_t* tiles, int x, int y) {
        if (x < 0 || y < 0 || x >= W || y >= H) return WALL_MID;
        return tiles[y + x * H];
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV_NOINLINE bool step(const State& s, const CommonState& c, int env, int action, float* reward, const StepCtx& ctx) {
        const int N = s.N;
        const uint8_t* tiles = s.tiles + (size_t)env * TILE_STRIDE;
        const float dt = 1.0f / SUB_STEPS;
        const int nspikes = s.num_spikes[env];
        auto tile_at = [&](int x, int y) { return get(tiles, x, H - 1 - y); };
        auto wall = [](int id) { return (id == WALL_MID || id == WALL_TOP) ? COLL_FULL : COLL_NONE; };

        float ax = s.ax[env], ay = s.ay[env], avx = s.avx[env], avy = s.avy[env], agent_t = s.agent_t[env];
        bool on_ground = s.on_ground[env] != 0, face_forward = s.face_forward[env] != 0;
        float jump_timer = s.jump_timer[env];
        int jumps_left = s.jumps_left[env];
        float cam_x = c.cam_x[env], cam_y = c.cam_y[env];
        float p_timer = s.p_timer[env];
        bool p_enabled = s.p_enabled[env] != 0;
        const float goal_x = s.goal_x[env], goal_y = s.goal_y[env];
        float to_goal_x = s.to_goal_x[env], to_goal_y = s.to_goal_y[env];
        const Rect goal_rect{ __fadd_rn(goal_x, -0.5f), __fadd_rn(goal_y, -0.5f), 1.0f, 1.0f };

        const float max_jump = 0.92f, gravity = 0.1f, max_speed = 0.5f, mix = 0.2f, air_control = 1.0f;
        const float movement_x = (float)((action == 6 || action == 7 || action == 8) - (action == 0 || action == 1 || action == 2));
        const bool jump = (action == 2 || action == 5 || action == 8);

        bool alive = true, achieved_goal = false;
        for (int ss = 0; ss < SUB_STEPS; ss++) {
            alive = true; achieved_goal = false;
            // ---- System_Agent::update
            {
                float mix_x = on_ground ? mix : __fmul_rn(mix, air_control);
                avx = __fadd_rn(avx, __fmul_rn(__fmul_rn(mix_x, __fsub_rn(__fmul_rn(max_speed, movement_x), avx)), dt));
                if (fabsf(avx) < __fmul_rn(__fmul_rn(mix_x, max_speed), dt)) avx = 0.0f;
                if (on_ground) jumps_left = 2;
                if (jump && jumps_left > 0 && jump_timer == 0.0f) { avy = -max_jump; jumps_left--; jump_timer = 3.0f; }
                if (jump_timer > 0.0f) jump_timer = fmaxf(0.0f, __fsub_rn(jump_timer, dt));
                avy = __fadd_rn(avy, __fmul_rn(gravity, dt));
                if (fabsf(avy) > max_jump) avy = __fmul_rn(avy > 0.0f ? 1.0f : -1.0f, max_jump);
                ax = __fadd_rn(ax, __fmul_rn(avx, dt));
                ay = __fadd_rn(ay, __fmul_rn(avy, dt));
                Rect world{ __fadd_rn(ax, -0.25f), __fadd_rn(ay, -0.8f), 0.5f, 0.8f };
                CollisionResult cd = tile_collision(world, tile_at, wall);
                float dpx = __fsub_rn(cd.x, world.x), dpy = __fsub_rn(cd.y, world.y);
                on_ground = dpy < 0.0f && cd.collided;
                ax = __fsub_rn(cd.x, -0.25f);
                ay = __fsub_rn(cd.y, -0.8f);
                world.x = __fadd_rn(ax, -0.25f); world.y = __fadd_rn(ay, -0.8f);
                if (dpx != 0.0f) avx = 0.0f;
                if (dpy > 0.0f && cd.collided) avy = 0.0f;
                if (on_ground) avy = 0.0f;
                bool hit = false;
                for (int k = ctx.lane; k < nspikes; k += ctx.nlanes) {
                    int cell = s.spike_cell[k * N + env];
                    float sx = __fadd_rn((float)(cell / H), 0.5f), sy = __fadd_rn((float)(H - 1 - cell % H), 0.5f);
                    Rect hz{ __fadd_rn(sx, -0.25f), __fadd_rn(sy, -0.25f), 0.5f, 0.5f };
                    if (check_collision(world, hz)) hit = true;
                }
                if (ctx.any(hit)) alive = false;
                if (check_collision(world, goal_rect)) achieved_goal = true;
                cam_x = __fmul_rn(ax, UNIT_TO_PIXELS);
                cam_y = __fmul_rn(__fsub_rn(ay, 0.5f), UNIT_TO_PIXELS);
                agent_t = __fadd_rn(agent_t, __fmul_rn(0.1f, dt));
                agent_t = fmodf(agent_t, 1.0f);
                if (movement_x > 0.0f) face_forward = true;
                else if (movement_x < 0.0f) face_forward = false;
                to_goal_x = __fsub_rn(goal_x, ax);
                to_goal_y = __fsub_rn(goal_y, ay);
                p_enabled = !on_ground || fabsf(avx) > 0.01f;
            }
            // ---- System_Particles::update (offset { 0.0f, -0.2f }, lifespan 5, spawn_time 0.5): one particle per lane
            {
                bool dead_here = false;
                for (int i = ctx.lane; i < NPART; i += ctx.nlanes) {
                    float life = __fsub_rn(s.p_life[i * N + env], dt);
                    s.p_life[i * N + env] = life;
                    if (life <= 0.0f) dead_here = true;
                }
                // dead_index = the LAST dead particle in index order
                int dead_index = -1;
                if (ctx.nlanes == 1) {
                    for (int i = 0; i < NPART; i++) if (s.p_life[i * N + env] <= 0.0f) dead_index = i;
                } else {
                    uint32_t m = __ballot_sync(0xffffffffu, dead_here && ctx.lane < NPART);
                    dead_index = m ? 31 - __clz(m) : -1;
                }
                p_timer = __fadd_rn(p_timer, dt);
                if (dead_index != -1 && p_timer >= 0.5f && p_enabled) {
                    p_timer = fmodf(p_timer, 0.5f);
                    int pi = dead_index * N + env;
                    if (ctx.leader()) {
                        s.p_life[pi] = 5.0f;
                        s.p_x[pi] = __fadd_rn(ax, 0.0f);
                        s.p_y[pi] = __fadd_rn(ay, -0.2f);
                    }
                }
                ctx.sync();
            }
            if (!alive || achieved_goal) break;
        }

        if (ctx.leader()) {
            s.ax[env] = ax; s.ay[env] = ay; s.avx[env] = avx; s.avy[env] = avy; s.agent_t[env] = agent_t;
            s.on_ground[env] = on_ground; s.face_forward[env] = face_forward;
            s.jump_timer[env] = jump_timer; s.jumps_left[env] = jumps_left;
            s.to_goal_x[env] = to_goal_x; s.to_goal_y[env] = to_goal_y;
            s.p_timer[env] = p_timer; s.p_enabled[env] = p_enabled;
            c.cam_x[env] = cam_x; c.cam_y[env] = cam_y;
            c.sprites_valid[env] = 1;
        }
        *reward = __fmul_rn((float)achieved_goal, 10.0f);
        return !alive || achieved_goal;
    }

    // ---------------------------------------------------------------------------------------
    struct Map {   // System_Tilemap helpers on the level-generation scratch (tilemap.cpp:54-77)
        uint8_t* t;
        PG2_DEV int get(int x, int y) const { return (x < 0 || y < 0 || x >= W || y >= H) ? (int)WALL_MID : (int)t[y + x * H]; }
        PG2_DEV void set(int x, int y, int id) { if (x < 0 || y < 0 || x >= W || y >= H) return; t[y + x * H] = (uint8_t)id; }
        PG2_DEV bool space_on_ground(int x, int y) const {
            if (get(x, y) != EMPTY) return false;
            if (get(x, y + 1) != EMPTY) return false;
            int below = get(x, y - 1);
            return below == WALL_MID || below == WALL_TOP;
        }
        PG2_DEV bool top_wall(int x, int y) const { return get(x, y) == WALL_MID && get(x, y + 1) == EMPTY; }
        PG2_DEV bool left_wall(int x, int y) const { return get(x, y) == WALL_MID && get(x + 1, y) == EMPTY; }
        PG2_DEV bool right_wall(int x, int y) const { return get(x, y) == WALL_MID && get(x - 1, y) == EMPTY; }
    };

    static PG2_DEV_NOINLINE void regenerate(const State& s, const CommonState& c, int env, WarpCtx& w) {
        const int N = s.N, lane = w.lane;
        bool fault = false;
        // ---- Maze_Generator::generate_maze_no_dead_ends(13, 13) (maze_generator.cpp:132-173)
        const int maze_scale = 3, maze_dim = W / maze_scale;
        MazeGrid mg = kruskal_maze(w, maze_dim, maze_dim);
        {
            const int ah = mg.ah, asize = mg.aw * mg.ah;
            for (int i = 0; i < asize; i++) {
                if (mg.grid[i] != 0) continue;
                const int x = i / ah, y = i % ah;
                const int nb[4] = { y + ah * (x - 1), y + ah * (x + 1), (y - 1) + ah * x, (y + 1) + ah * x };
                int spaces = 0, walls = 0;
                for (int n = 0; n < 4; n++) { int v = mg.grid[nb[n]]; spaces += v == 0; walls += v == 1; }
                if (spaces == 1 && walls > 0) {
                    int n_select = w.rng.uniform_int(0, walls - 1);
                    __syncwarp();
                    for (int n = 0; n < 4; n++) {
                        int cell = nb[(n_select + n) % walls];   // indexes ALL neighbours, not only walls (SURVEY Q6)
                        int cx = cell / ah, cy = cell % ah;
                        if (cx >= 1 && cy >= 1 && cx < mg.aw - 1 && cy < mg.ah - 1 && mg.grid[cell] == 1) { mg.grid[cell] = 0; break; }
                    }
                    __syncwarp();
                }
            }
        }
        RoomGen rg;
        rg.init(w, W, H);
        uint8_t* tiles = w.alloc<uint8_t>((W * H + 3) & ~3);
        uint16_t* cand = rg.parents;                   // agent_candidates (before find_path reuses the buffer)
        uint16_t* spikes = w.alloc<uint16_t>(MAX_SPIKES);
        uint8_t* order = w.alloc<uint8_t>(MAX_SPIKES + 8);
        USet<MAX_SPIKES + 8, 128>* us = w.alloc<USet<MAX_SPIKES + 8, 128>>(1);
        Map map{ tiles };

        w.rng.bernoulli_fill(rg.grid, W * H, [&](int i) {   // wall with probability 0.8 under a maze wall, else 0.2
            int obj = mg.grid[((i % H) / maze_scale + 1) + mg.ah * ((i / H) / maze_scale + 1)];
            return obj == 1 ? 0.8f : 0.2f;
        });
        rg.update(w);
        rg.update(w);
        for (int i = lane; i < W; i += WARP_LANES) {
            rg.grid[0 + H * i] = 1; rg.grid[(H - 1) + H * i] = 1;      // set(i, 0), set(i, H-1)
            rg.grid[i + H * 0] = 1; rg.grid[i + H * (W - 1)] = 1;      // set(0, i), set(W-1, i)
        }
        int nroom = rg.find_best_room(w);
        if (nroom <= 0) { fault = true; nroom = 1; rg.order[0] = (uint16_t)(1 + H); }
        for (int i = lane; i < W * H; i += WARP_LANES) tiles[i] = WALL_MID;
        __syncwarp();
        for (int i = lane; i < nroom; i += WARP_LANES) tiles[rg.order[i]] = EMPTY;
        __syncwarp();
        const int goal_cell = rg.order[w.rng.uniform_int(0, nroom - 1)];

        int ncand = warp_compact(w, W * H, [&](int i) { return map.space_on_ground(i / H, i % H) && i != goal_cell; }, cand);
        if (ncand <= 0) { fault = true; ncand = 1; if (lane == 0) cand[0] = rg.order[0]; __syncwarp(); }   // Q20
        const int agent_cell = cand[w.rng.uniform_int(0, ncand - 1)];
        __syncwarp();

        if (PRUNE) {   // only wide_path = goal_path dilated 4 times stays open (find_path draws nothing: skipped otherwise)
            int plen = rg.find_path(w, agent_cell, goal_cell);
            rg.expand(w, rg.path, plen, 4, rg.mark);
            for (int i = lane; i < W * H; i += WARP_LANES) tiles[i] = rg.mark[i] ? EMPTY : WALL_MID;
            __syncwarp();
        }

        const float goal_x = __fadd_rn((float)(goal_cell / H), 0.5f), goal_y = __fadd_rn((float)(H - 1 - goal_cell % H), 0.5f);

        // spikes, then wall thinning: scans whose writes feed later tests, RNG draws inside -> uniform serial code
        {   // a spike only turns EMPTY cells non-empty, which can only falsify later tests: the cells passing the test on
            // the spike-free map (lane-parallel scan, x-major order kept) are a superset; re-check those in order
            uint16_t* sc = rg.queue;
            int nsc = warp_compact(w, W * H, [&](int i) {
                int x = i / H, y = i % H;
                return map.space_on_ground(x, y) && map.space_on_ground(x - 1, y) && map.space_on_ground(x + 1, y); }, sc);
            for (int k = 0; k < nsc; k++) {
                int x = sc[k] / H, y = sc[k] % H;
                if (map.space_on_ground(x, y) && map.space_on_ground(x - 1, y) && map.space_on_ground(x + 1, y)) {
                    bool put = w.rng.uniform_real(0.0f, 1.0f) < SPIKE_PROB;
                    __syncwarp();
                    if (put) map.set(x, y, SPIKE);
                    __syncwarp();
                }
            }
        }
        // wall thinning (tilemap.cpp): cells in x-major order, per cell the left test then the right test, every hit
        // draws from the RNG and clears a wall cell — which can enable as well as disable later tests. The warp tests
        // 32 cells at a time on the CURRENT map, serves the first hit in order, and resumes right behind it.
        {
            int pos = 0, skip_left = 0;   // next cell to test; skip_left: its left test has been served already
            while (pos < W * H) {
                const int i = pos + lane, x = i / H, y = i % H;
                const bool in = i < W * H;
                const bool hl = in && !(lane == 0 && skip_left) && map.left_wall(x, y) && map.left_wall(x, y + 1) && map.left_wall(x, y + 2);
                const bool hr = in && map.right_wall(x, y) && map.right_wall(x, y + 1) && map.right_wall(x, y + 2);
                const uint32_t ml = lane_ballot(hl, lane), mr = lane_ballot(hr, lane);
                if (!(ml | mr)) { pos += WARP_LANES; skip_left = 0; continue; }
                const int l = __ffs(ml | mr) - 1, hit = pos + l, hx = hit / H, hy = hit % H;
                const bool left = (ml >> l) & 1u;
                int d = w.rng.uniform_int(0, 2);
                __syncwarp();
                map.set(hx, hy + d, EMPTY);
                __syncwarp();
                if (left) { pos = hit; skip_left = 1; } else { pos = hit + 1; skip_left = 0; }
            }
        }
        const float agent_x = __fadd_rn((float)(agent_cell / H), 0.5f), agent_y = (float)(H - 1 - (agent_cell % H));

        int nspikes = warp_compact(w, W * H, [&](int i) { return tiles[i] == SPIKE && i != agent_cell && i != goal_cell; }, rg.queue);
        if (nspikes > MAX_SPIKES) { fault = true; nspikes = MAX_SPIKES; }
        for (int k = lane; k < nspikes; k += WARP_LANES) spikes[k] = rg.queue[k];
        __syncwarp();
        for (int i = lane; i < W * H; i += WARP_LANES) if (tiles[i] == SPIKE) tiles[i] = EMPTY;
        __syncwarp();
        // tops (order-insensitive: a cell turned into wall_top is neither wall_mid nor empty for its neighbours' tests)
        for (int i = lane; i < W * H; i += WARP_LANES) rg.tmp[i] = map.top_wall(i / H, i % H) ? 1 : 0;
        __syncwarp();
        for (int i = lane; i < W * H; i += WARP_LANES) if (rg.tmp[i]) tiles[i] = WALL_TOP;
        __syncwarp();

        // ---- reset() tail
        int bg_index = w.rng.uniform_int(0, PG2_NUM_PLATFORM_BACKGROUNDS - 1);
        float bg_offset = w.rng.uniform_real(0.0f, 1.0f);
        int map_theme = w.rng.uniform_int(0, 3);

        // sprite_render set: goal (id 0), spikes (ids 2..)
        us->init(s.nb_sprite[env]);
        us->insert(0);
        for (int k = 0; k < nspikes; k++) us->insert(2 + k);
        int nsp = us->order(order);
        int nb_sprite = us->nb;
        __syncwarp();
        for (int k = lane; k < nsp; k += WARP_LANES) s.sprite_order[k * N + env] = (uint8_t)(order[k] == 0 ? 0 : order[k] - 1);

        uint8_t* gt = s.tiles + (size_t)env * TILE_STRIDE;
        for (int i = lane; i < (W * H + 3) / 4; i += WARP_LANES) ((uint32_t*)gt)[i] = ((const uint32_t*)tiles)[i];   // (the scratch map is padded to a word)
        for (int k = lane; k < nspikes; k += WARP_LANES) s.spike_cell[k * N + env] = spikes[k];
        for (int k = lane; k < NPART; k += WARP_LANES) { s.p_x[k * N + env] = 0.0f; s.p_y[k * N + env] = 0.0f; s.p_life[k * N + env] = 0.0f; }
        if (lane == 0) {
            s.num_spikes[env] = nspikes;
            s.nb_sprite[env] = nb_sprite;
            s.goal_x[env] = goal_x; s.goal_y[env] = goal_y;
            s.ax[env] = agent_x; s.ay[env] = agent_y; s.avx[env] = 0.0f; s.avy[env] = 0.0f;
            s.on_ground[env] = 0; s.face_forward[env] = 1; s.agent_t[env] = 0.0f;
            s.jump_timer[env] = 0.0f; s.jumps_left[env] = 2;
            s.p_timer[env] = 0.0f; s.p_enabled[env] = 1;
            s.bg_index[env] = bg_index; s.bg_offset[env] = bg_offset; s.map_theme[env] = map_theme;
            c.sprites_valid[env] = 0;
            if (fault) c.fault[env] |= 1;
        }
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV int tile_class(uint32_t tex) { return tex < (uint32_t)T_WALL_MID0 ? 1 : 0; }

    template <class F>
    static PG2_DEV_NOINLINE void build_frame(const State& s, const CommonState& c, int env, F& f, const TexInfo* tex) {
        const int N = s.N;
        const float zoom = 0.3f;
        Camera cam{ c.cam_x[env], c.cam_y[env], __fdiv_rn(__fmul_rn(zoom, f.view_w), 64.0f), f.view_w, f.view_h };
        int lx, ly, ux, uy;
        tile_window(cam, &lx, &ly, &ux, &uy);
        const int ncol = min(ux - lx + 1, MAX_WIN), nrow = min(uy - ly + 1, MAX_WIN);
        const int nspikes = s.num_spikes[env];
        const int nspr = c.sprites_valid[env] ? nspikes + 1 : 0;
        const int theme = s.map_theme[env];
        // background (e.g. maze.cpp:402-408): the blit itself is built by build_tile_layer below
        const int bg = T_BG0 + s.bg_index[env];
        const TexInfo bt = tex[bg];
        const float bg_x = __fmul_rn(-s.bg_offset[env], __fsub_rn(__fdiv_rn((float)bt.w, (float)bt.h), 1.0f));
        const float bg_scale = __fdiv_rn(__fmul_rn(64.0f, UNIT_TO_PIXELS), (float)bt.h);
        const int o_spr = NPART, o_agent = o_spr + nspr, o_hud = o_agent + 1;
        // tile layer: class 0 = wall_mid texture of the theme, class 1 = wall_top texture
        const uint8_t* tiles = s.tiles + (size_t)env * TILE_STRIDE;
        build_tile_layer(f, cam, tex, 2, lx, ly, ncol, nrow, [&](int cls) { return (cls ? T_WALL_TOP0 : T_WALL_MID0) + theme; }, [&](int x, int y) {
            const int id = get(tiles, x, H - 1 - y);
            return id == WALL_MID ? T_WALL_MID0 + theme : id == WALL_TOP ? T_WALL_TOP0 + theme : (int)NO_TILE;
        }, bg, bg_x, 0.0f, bg_scale);
        emit_post_blits(f, tex, o_hud + 3, [&](int k, BlitReq& b, BlitRot& rot) {
            if (k < o_spr) {   // System_Particles::render
                int pi = k * N + env;
                float life = s.p_life[pi];
                if (life <= 0.0f) return;
                float life_ratio = __fdiv_rn(__fsub_rn(5.0f, life), 5.0f);
                float alpha = __fmul_rn(0.5f, __fsub_rn(1.0f, life_ratio));
                float scale = __fmul_rn(0.45f, __fadd_rn(__fmul_rn(0.4f, life_ratio), 0.6f));
                float offset_y = __fmul_rn(-life_ratio, 0.17f);
                float pw = (float)tex[T_PARTICLE].w, ph = (float)tex[T_PARTICLE].h;
                float px = __fsub_rn(__fmul_rn(s.p_x[pi], UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(0.5f, pw), scale));
                float py = __fsub_rn(__fmul_rn(__fadd_rn(s.p_y[pi], offset_y), UNIT_TO_PIXELS), __fmul_rn(__fmul_rn(0.5f, ph), scale));
                b.plain(T_PARTICLE, px, py, cam, __fdiv_rn(__fmul_rn(scale, UNIT_TO_PIXELS), pw), alpha);
            } else if (k < o_agent) {
                int sp = s.sprite_order[sort_perm(nspr, k - o_spr) * N + env];
                if (sp == 0) {
                    float px = __fmul_rn(__fadd_rn(s.goal_x[env], -0.5f), UNIT_TO_PIXELS);
                    float py = __fmul_rn(__fadd_rn(s.goal_y[env], -0.5f), UNIT_TO_PIXELS);
                    b.plain(T_CARROT, px, py, cam, __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, 1.0f), UNIT_TO_PIXELS), (float)tex[T_CARROT].w));
                } else {
                    int cell = s.spike_cell[(sp - 1) * N + env];
                    float sx = __fadd_rn((float)(cell / H), 0.5f), sy = __fadd_rn((float)(H - 1 - cell % H), 0.5f);
                    float px = __fmul_rn(__fadd_rn(sx, -0.25f), UNIT_TO_PIXELS);
                    float py = __fmul_rn(__fadd_rn(sy, -0.25f), UNIT_TO_PIXELS);
                    b.plain(T_SPIKE, px, py, cam, __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, 0.4f), UNIT_TO_PIXELS), (float)tex[T_SPIKE].w));
                }
            } else if (k == o_agent) {   // System_Agent::render
                float avx = s.avx[env];
                bool on_ground = s.on_ground[env] != 0;
                int t; float agent_scale = 0.5f, off_x = 0.0f, off_y = 0.2f;
                if (fabsf(avx) < 0.01f && on_ground) t = T_STAND;
                else if (!on_ground) { t = T_JUMP; agent_scale = 0.6f; off_x = -0.05f; off_y = 0.25f; }
                else if (s.agent_t[env] > 0.5f) t = T_WALK2;
                else t = T_WALK1;
                float posx = __fsub_rn(s.ax[env], 0.25f), posy = __fsub_rn(s.ay[env], 1.0f);
                float px = __fmul_rn(__fadd_rn(posx, off_x), UNIT_TO_PIXELS);
                float py = __fmul_rn(__fadd_rn(posy, off_y), UNIT_TO_PIXELS);
                b.plain(t, px, py, cam, __fmul_rn(__fdiv_rn(UNIT_TO_PIXELS, (float)tex[t].w), agent_scale), 1.0f, s.face_forward[env] == 0);
            } else {   // compass HUD (jumper.cpp:474-509), obs target: width = 64, game_zoom = 0.3
                const float compass_size = 200.0f, off_x = -32.0f, off_y = 32.0f, width = f.view_w;   // (the HUD keeps game_zoom: it does not scale with the window)
                const float tgx = s.to_goal_x[env], tgy = s.to_goal_y[env];
                float dist = __fsqrt_rn(__fadd_rn(__fmul_rn(tgx, tgx), __fmul_rn(tgy, tgy)));
                if (k == o_hud) {
                    b.rect(T_CIRCLE, __fadd_rn(__fsub_rn(width, __fmul_rn(compass_size, zoom)), __fmul_rn(off_x, zoom)),
                                       __fmul_rn(off_y, zoom), __fmul_rn(compass_size, zoom), __fmul_rn(compass_size, zoom), 0.0, &rot);
                } else if (k == o_hud + 1) {
                    float angle = (float)__ddiv_rn((double)__fmul_rn(glibc_atan2f(tgy, tgx), 180.0f), 3.14159265358979323846);
                    float dist_inv = __fdiv_rn(1.0f, fmaxf(0.0001f, dist));
                    float dir_x = __fmul_rn(tgx, dist_inv), dir_y = __fmul_rn(tgy, dist_inv);
                    float x = __fadd_rn(__fsub_rn(width, __fmul_rn(__fmul_rn(compass_size, 0.75f), zoom)), __fmul_rn(off_x, zoom));
                    float y = __fadd_rn(__fmul_rn(__fmul_rn(compass_size, 0.5f), zoom), __fmul_rn(off_y, zoom));
                    x = __fadd_rn(x, __fmul_rn(__fmul_rn(__fmul_rn(compass_size, 0.25f), dir_x), zoom));
                    y = __fadd_rn(y, __fmul_rn(__fmul_rn(__fmul_rn(compass_size, 0.25f), dir_y), zoom));
                    b.rect(T_NEEDLE, x, y, __fmul_rn(__fmul_rn(compass_size, 0.5f), zoom),
                                       __fmul_rn(__fmul_rn(compass_size, 0.1f), zoom), (double)angle, &rot);
                } else {
                    float ratio = fminf(1.0f, __fdiv_rn(dist, __fmul_rn((float)W, 1.414f)));
                    b.rect(T_BAR, __fadd_rn(__fsub_rn(width, __fmul_rn(compass_size, zoom)), __fmul_rn(off_x, zoom)),
                                       __fadd_rn(__fmul_rn(compass_size, zoom), __fmul_rn(off_y, zoom)),
                                       __fmul_rn(__fmul_rn(compass_size, zoom), ratio), __fmul_rn(__fmul_rn(compass_size, 0.15f), zoom), 0.0, &rot);
                }
            }
        });
    }
};
using Jumper = JumperT<1>;

}  // namespace pg2
