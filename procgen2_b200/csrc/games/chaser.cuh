// Chaser — device restatement of /root/reference/games/chaser/:
//   step logic  cenv_step chaser.cpp:282-320; System_Agent::update common_systems.cpp:305-444;
//               System_Mob_AI::update :117-295 (eat :297); System_Point::update :66-106;
//               System_Sprite_Render::update :8-40
//   level gen   System_Tilemap::regenerate tilemap.cpp:80-243 (spawn helpers :30-78),
//               Maze_Generator::generate_maze maze_generator.cpp:47-130, reset() chaser.cpp:420-447
//   frame       render_game chaser.cpp:390-418; tilemap.cpp:245-267; common_systems.cpp:42-64, 446-462
// All three distribution modes of tilemap.cpp:85-99 as ChaserT<MODE>: 0 easy (the reference's compiled-in default,
// tilemap.h:40): 11 x 11 world, 3 enemies, 4 orbs; 1 hard: 13 x 13, 3 enemies, 3 orbs (one quadrant has none);
// 2 extreme: 19 x 19, 5 enemies, 5 orbs (one quadrant has two).
// Entity ids per episode (SURVEY App. B), easy: 0-3 orbs, 4-6 eggs, 7-69 points, 70 agent (orbs, eggs, points, agent in
// creation order in every mode).
// abs() on floats is the float overload (SURVEY Q16).
#pragma once
#include "../pg2_common.cuh"
#include "../pg2_mazegen.cuh"
#include "../pg2_render.cuh"
#include "../pg2_rng.cuh"
#include "../pg2_state.cuh"
#include "../pg2_uset.cuh"
#include "../pg2_warp.cuh"

namespace pg2 {

// CELL: type of a cell index y + x*H (19 x 19 needs 16 bits); NT / NF / NE / NM: capacities of the tile map, the point
// cells, the sprite entities and the mobs
#define PG2_CHASER_FIELDS_(F, CELL, NT, NF, NE, NM)                                                \
    PG2_ENV_MAJOR(F)(uint8_t, tiles, NT) /* [y + x*H]: 0 empty, 1 wall */                          \
    PG2_ENV_MAJOR(F)(CELL, free_cells, NF) /* System_Tilemap::free_cells after regenerate (the point cells) */ \
    F(int32_t, num_free, 1)                                                                       \
    F(int32_t, num_ents, 1)     /* sprite entities: orbs, eggs, points */                         \
    F(uint8_t, ent_kind, NE)    /* slot-major: 1 orb, 2 egg/mob, 3 point, 0 destroyed */          \
    F(CELL, ent_cell, NE)       /* spawn cell index (y + x*H, map space) of orbs and points */    \
    F(uint8_t, sprite_order, NE) /* iteration order of System_Sprite_Render::entities at reset */ \
    F(uint8_t, mob_order, NM + 1) /* iteration order of System_Mob_AI::entities (mob slots 0..NM-1) */ \
    F(int32_t, nb_sprite, 1) F(int32_t, nb_mob, 1)   /* persisted bucket counts (Q25) */           \
    F(float, mob_x, NM) F(float, mob_y, NM) F(float, mob_vx, NM) F(float, mob_vy, NM)              \
    F(float, mob_hatch, NM) F(uint8_t, mob_tex, NM)                                                \
    F(float, anim_timer, 1) F(int32_t, anim_index, 1) F(float, eat_timer, 1)                       \
    F(float, ax, 1) F(float, ay, 1) F(float, avx, 1) F(float, avy, 1)                              \
    F(float, next_vx, 1) F(float, next_vy, 1) F(float, input_timer, 1)                             \
    F(int32_t, bg_index, 1) F(float, bg_offset, 1)
#define PG2_CHASER_FIELDS(F) PG2_CHASER_FIELDS_(F, uint8_t, 128, 64, 72, 3)
#define PG2_CHASER_FIELDS_HARD(F) PG2_CHASER_FIELDS_(F, uint8_t, 256, 128, 104, 3)
#define PG2_CHASER_FIELDS_EXTREME(F) PG2_CHASER_FIELDS_(F, uint16_t, 384, 256, 208, 5)

PG2_DEFINE_STATE(ChaserState, PG2_CHASER_FIELDS)
PG2_DEFINE_STATE(ChaserStateHard, PG2_CHASER_FIELDS_HARD)
PG2_DEFINE_STATE(ChaserStateExtreme, PG2_CHASER_FIELDS_EXTREME)
template <int MODE> struct ChaserStateOf { using type = ChaserState; using cell_t = uint8_t; };
template <> struct ChaserStateOf<1> { using type = ChaserStateHard; using cell_t = uint8_t; };
template <> struct ChaserStateOf<2> { using type = ChaserStateExtreme; using cell_t = uint16_t; };

template <int MODE>
struct ChaserT {
    using State = typename ChaserStateOf<MODE>::type;
    using cell_t = typename ChaserStateOf<MODE>::cell_t;
    static constexpr int W = MODE == 1 ? 13 : MODE == 2 ? 19 : 11, H = W;   // world_dim (tilemap.cpp:85-99)
    static constexpr int NMOB = MODE == 2 ? 5 : 3;                          // total_enemies
    static constexpr int ORB_SIGN = MODE == 1 ? -1 : MODE == 2 ? 1 : 0;     // extra_orb_sign: orbs of the one "extra" quadrant
    static constexpr int NORB = 4 + ORB_SIGN;                               // orbs = the first entity ids, the eggs follow
    static constexpr int MAX_ENTS = MODE == 1 ? 104 : MODE == 2 ? 208 : 72; // orbs + eggs + points (70 / 96 / 198 in every level seen)
    static constexpr int QUAD_CAP = MODE == 2 ? 128 : 64;                   // free cells of one quadrant
    static constexpr int FC_CAP = MODE == 2 ? 256 : 128;                    // free cells of the world
    using Set = USet<(MODE == 2 ? 256 : 128), (MODE == 2 ? 264 : 128)>;
    static constexpr int SUB_STEPS = 4;
    static constexpr bool LANE_AWARE = true;    // step(): the point loop is strided over ctx's lanes, the rest is uniform
    static constexpr int STEP_LANES = 32;       // lanes per environment in k_step
    static constexpr int MAX_POST = MODE == 1 ? 104 : MODE == 2 ? 208 : 80;   // capacity of the frame's post-blit list
    static constexpr bool ROTATES = false;     // some blits are rotated
    static constexpr bool SLOW_RESET = true;    // level generation (Kruskal + set orders, ~0.1 ms) runs concurrently with the render of the other envs: +22 % at 4096 envs
    static constexpr int RESET_ARENA = (MODE == 1 ? 6 : MODE == 2 ? 10 : 4) * 1024;   // per-warp level-generation scratch (high water measured with PG2_ARENA_TRACE)
    static constexpr bool PREFETCH_LEVELS = false;   // step() draws from the RNG: the next level is not known ahead of time
    static constexpr int PREFETCH_MIN_EPISODE = 0;   // level prefetch whatever max_episode_steps is
    static const char* reset_keeps() { return ""; }
    static constexpr int TILE_CLASSES = 1;
    static constexpr int WIN_ROWS = MODE == 1 ? 16 : MODE == 2 ? 22 : 14;        // most tile rows the camera window can span (zoom-dependent; frame table sizing)
    static constexpr int BLIT_UNROLL = 1;     // post-blit patches fetched together (pg2_render.cuh draw_blit_band)
    static constexpr int RENDER_MIN_CTAS = 8;   // CTAs per SM the register allocation of k_render aims at
    static constexpr int DEFAULT_MODE = MODE;    // this instantiation's distribution mode (the reference compiles in 0 = easy; tilemap.h Config)
    static bool mode_supported(int mode) { return mode == MODE; }
    static constexpr bool HAS_TILES = true;     // the frame has a tile layer
    static constexpr bool STATIC_VIEW = true;    // fixed camera and tile map within an episode: the base image (background + tiles) is cached per env
    static constexpr int TILE_STRIDE = MODE == 1 ? 256 : MODE == 2 ? 384 : 128, FREE_STRIDE = MODE == 1 ? 128 : MODE == 2 ? 256 : 64;
    enum Kind { K_NONE = 0, K_ORB, K_MOB, K_POINT };
    enum Tex { T_WALL = 0, T_CRYSTAL, T_EGG, T_POINT, T_FLY0, T_FLY1, T_FLY2, T_WALK, T_AGENT, T_BG0, NUM_BG = 9, NUM_TEX = 18 };

    static const char* const* texture_names(int* count) {
        static const char* const names[NUM_TEX] = {
            "assets/misc_assets/tileStone_slope.png", "assets/misc_assets/yellowCrystal.png",
            "assets/misc_assets/enemySpikey_1b.png", "assets/custom/chaser_point.png",
            "assets/misc_assets/enemyFlying_1.png", "assets/misc_assets/enemyFlying_2.png",
            "assets/misc_assets/enemyFlying_3.png", "assets/misc_assets/enemyWalking_1b.png",
            "assets/misc_assets/enemyFloating_1b.png",
            "assets/topdown_backgrounds/floortiles.png",
            "assets/topdown_backgrounds/backgrounddetailed1.png", "assets/topdown_backgrounds/backgrounddetailed2.png",
            "assets/topdown_backgrounds/backgrounddetailed3.png", "assets/topdown_backgrounds/backgrounddetailed4.png",
            "assets/topdown_backgrounds/backgrounddetailed5.png", "assets/topdown_backgrounds/backgrounddetailed6.png",
            "assets/topdown_backgrounds/backgrounddetailed7.png", "assets/topdown_backgrounds/backgrounddetailed8.png",
        };
        *count = NUM_TEX;
        return names;
    }

    // System_Tilemap::get (tilemap.h:78-83): out of bounds is `out_of_bounds` (-1), never `empty`.
    static PG2_DEV int get(const uint8_t* tiles, int x, int y) {
        if (x < 0 || y < 0 || x >= W || y >= H) return -1;
        return tiles[y + x * H];
    }
    static PG2_DEV int sign(float x) { return x == 0.0f ? 0 : (x > 0.0f) * 2 - 1; }   // helpers.h:31-36
    static PG2_DEV float cell_center(float v) { return __fadd_rn((float)f2i(v), 0.5f); }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV_NOINLINE bool step(const State& s, const CommonState& c, int env, int action, float* reward, const StepCtx& ctx) {
        const int N = s.N;
        const uint8_t* tiles = s.tiles + (size_t)env * TILE_STRIDE;
        const float dt = 1.0f / SUB_STEPS;
        Mt rng; rng.mt = c.mt + (size_t)env * MT_N; rng.idx = c.mti[env];
        const int nents = s.num_ents[env];

        float ax = s.ax[env], ay = s.ay[env], avx = s.avx[env], avy = s.avy[env];
        float next_vx = s.next_vx[env], next_vy = s.next_vy[env], input_timer = s.input_timer[env];
        float anim_timer = s.anim_timer[env], eat_timer = s.eat_timer[env];
        int anim_index = s.anim_index[env];

        const float speed = 0.2f;
        const float input_reset_time = __fmul_rn(__fdiv_rn(1.0f, speed), 0.5f);
        const float tol = __fmul_rn(speed, dt);
        float movement_x = (float)((action == 7) - (action == 1));
        float movement_y = (float)((action == 3) - (action == 5));
        if (movement_x != 0.0f && movement_y != 0.0f) movement_y = 0.0f;

        bool dead = false;
        int point_delta = 0, points_available = 0;
        for (int ss = 0; ss < SUB_STEPS; ss++) {
            // ================= System_Agent::update =================
            {
                if (movement_x != 0.0f || movement_y != 0.0f) { next_vx = movement_x; next_vy = movement_y; input_timer = 0.0f; }
                if (next_vx > 0.0f) {
                    if (fabsf(__fsub_rn(ay, cell_center(ay))) <= tol && get(tiles, f2i(ax) + 1, H - 1 - f2i(ay)) == 0) {
                        ay = cell_center(ay); avx = next_vx; avy = next_vy;
                    }
                } else if (next_vx < 0.0f) {
                    if (fabsf(__fsub_rn(ay, cell_center(ay))) <= tol && get(tiles, f2i(ax) - 1, H - 1 - f2i(ay)) == 0) {
                        ay = cell_center(ay); avx = next_vx; avy = next_vy;
                    }
                }
                if (next_vy > 0.0f) {
                    if (fabsf(__fsub_rn(ax, cell_center(ax))) <= tol && get(tiles, f2i(ax), H - 1 - (f2i(ay) + 1)) == 0) {
                        ax = cell_center(ax); avx = next_vx; avy = next_vy;
                    }
                } else if (next_vy < 0.0f) {
                    if (fabsf(__fsub_rn(ax, cell_center(ax))) <= tol && get(tiles, f2i(ax), H - 1 - (f2i(ay) - 1)) == 0) {
                        ax = cell_center(ax); avx = next_vx; avy = next_vy;
                    }
                }
                if (avx < 0.0f) {
                    if (fabsf(__fsub_rn(ax, cell_center(ax))) <= tol && get(tiles, f2i(ax) - 1, H - 1 - f2i(ay)) != 0) { ax = cell_center(ax); avx = 0.0f; }
                } else if (avx > 0.0f) {
                    if (fabsf(__fsub_rn(ax, cell_center(ax))) <= tol && get(tiles, f2i(ax) + 1, H - 1 - f2i(ay)) != 0) { ax = cell_center(ax); avx = 0.0f; }
                }
                if (avy < 0.0f) {
                    if (fabsf(__fsub_rn(ay, cell_center(ay))) <= tol && get(tiles, f2i(ax), H - 1 - (f2i(ay) - 1)) != 0) { ay = cell_center(ay); avy = 0.0f; }
                } else if (avy > 0.0f) {
                    if (fabsf(__fsub_rn(ay, cell_center(ay))) <= tol && get(tiles, f2i(ax), H - 1 - (f2i(ay) + 1)) != 0) { ay = cell_center(ay); avy = 0.0f; }
                }
                ax = __fadd_rn(ax, __fmul_rn(__fmul_rn(avx, speed), dt));
                ay = __fadd_rn(ay, __fmul_rn(__fmul_rn(avy, speed), dt));
                if (input_timer >= input_reset_time) { next_vx = 0.0f; next_vy = 0.0f; }
                else input_timer = __fadd_rn(input_timer, dt);
            }
            const Rect agent_rect{ __fadd_rn(-0.5f, ax), __fadd_rn(-0.5f, ay), 1.0f, 1.0f };

            // ================= System_Mob_AI::update =================
            dead = false;
            for (int k = 0; k < NMOB; k++) {
                const int m = s.mob_order[k * N + env];
                float hatch = s.mob_hatch[m * N + env];
                if (hatch >= 50.0f) {
                    float x = s.mob_x[m * N + env], y = s.mob_y[m * N + env], vx = s.mob_vx[m * N + env], vy = s.mob_vy[m * N + env];
                    int tex;
                    float mspeed;
                    if (eat_timer == 0.0f) { tex = anim_index < 3 ? T_FLY0 + anim_index : T_FLY0 + (5 - anim_index); mspeed = 0.25f; }
                    else { tex = T_WALK; mspeed = 0.125f; }
                    bool at_junction = fmaxf(fabsf(__fsub_rn(x, cell_center(x))), fabsf(__fsub_rn(y, cell_center(y)))) < __fmul_rn(mspeed, dt);
                    if ((vx == 0.0f && vy == 0.0f) || at_junction) {
                        bool poss[4];
                        int num = 0;
                        const int ix = f2i(x), iy = f2i(y);
                        poss[0] = get(tiles, ix - 1, H - 1 - iy) == 0 && -1 != -sign(vx);
                        poss[1] = get(tiles, ix + 1, H - 1 - iy) == 0 && 1 != -sign(vx);
                        poss[2] = get(tiles, ix, H - 1 - (iy - 1)) == 0 && -1 != -sign(vy);
                        poss[3] = get(tiles, ix, H - 1 - (iy + 1)) == 0 && 1 != -sign(vy);
                        for (int i = 0; i < 4; i++) num += poss[i];
                        const float dirx[4] = { -1.0f, 1.0f, 0.0f, 0.0f }, diry[4] = { 0.0f, 0.0f, -1.0f, 1.0f };
                        bool be_aggressive = rng.canonical() < 0.5f;
                        int sel = 0;
                        if (be_aggressive) {
                            float min_dist = 999999.0f;
                            for (int i = 0; i < 4; i++)
                                if (poss[i]) {
                                    float md = __fadd_rn(fabsf(__fsub_rn(__fadd_rn(x, dirx[i]), ax)), fabsf(__fsub_rn(__fadd_rn(y, diry[i]), ay)));
                                    if (eat_timer > 0.0f) md = -md;
                                    if (md < min_dist) { min_dist = md; sel = i; }
                                }
                        } else if (num > 0) {
                            int cusp = rng.uniform_int(0, num - 1);
                            int sum = 0;
                            for (int i = 0; i < 4; i++) { sum += poss[i]; if (sum > cusp) { sel = i; break; } }
                        }
                        vx = __fmul_rn(dirx[sel], mspeed);
                        vy = __fmul_rn(diry[sel], mspeed);
                        if (dirx[sel] == 0.0f) x = cell_center(x);
                        if (diry[sel] == 0.0f) y = cell_center(y);
                    }
                    x = __fadd_rn(x, __fmul_rn(vx, dt));
                    y = __fadd_rn(y, __fmul_rn(vy, dt));
                    Rect rect{ __fadd_rn(-0.5f, x), __fadd_rn(-0.5f, y), 1.0f, 1.0f };
                    if (check_collision(agent_rect, rect)) {
                        if (eat_timer == 0.0f) dead = true;
                        else {   // respawn as an egg; y is NOT flipped here (SURVEY Q17)
                            hatch = 0.0f;
                            int cell = s.free_cells[(size_t)env * FREE_STRIDE + rng.uniform_int(0, s.num_free[env] - 1)];
                            x = __fadd_rn((float)(cell / H), 0.5f);
                            y = __fadd_rn((float)(cell % H), 0.5f);
                            tex = T_EGG;
                        }
                    }
                    s.mob_x[m * N + env] = x; s.mob_y[m * N + env] = y; s.mob_vx[m * N + env] = vx; s.mob_vy[m * N + env] = vy;
                    s.mob_tex[m * N + env] = (uint8_t)tex;
                } else {
                    hatch = __fadd_rn(hatch, dt);
                }
                s.mob_hatch[m * N + env] = hatch;
            }
            if (anim_timer < 1.0f) anim_timer = __fadd_rn(anim_timer, dt);
            else { anim_timer = __fsub_rn(anim_timer, 1.0f); anim_index = (anim_index + 1) % 6; }
            if (eat_timer > 0.0f) eat_timer = fmaxf(0.0f, __fsub_rn(eat_timer, dt));

            // ================= System_Point::update =================
            ctx.sync();
            int delta = 0, avail = 0;
            bool ate_orb = false;
            for (int e = ctx.lane; e < nents; e += ctx.nlanes) {
                int kind = s.ent_kind[e * N + env];
                if (kind != K_ORB && kind != K_POINT) continue;
                int cell = s.ent_cell[e * N + env];
                float px = __fadd_rn((float)(cell / H), 0.5f), py = __fadd_rn((float)(H - 1 - cell % H), 0.5f);
                Rect rect = kind == K_ORB ? Rect{ __fadd_rn(-0.5f, px), __fadd_rn(-0.5f, py), 1.0f, 1.0f }
                                          : Rect{ __fadd_rn(-0.3f, px), __fadd_rn(-0.3f, py), 0.6f, 0.6f };
                if (check_collision(agent_rect, rect)) {
                    if (kind == K_ORB) ate_orb = true;
                    delta++;
                    s.ent_kind[e * N + env] = K_NONE;
                } else avail++;
            }
            if (ctx.any(ate_orb)) eat_timer = 75.0f;   // System_Mob_AI::eat()
            point_delta = ctx.sum(delta);
            points_available = ctx.sum(avail);
            if (dead || points_available == 0) break;
        }

        ctx.sync();
        if (ctx.leader()) {
            s.ax[env] = ax; s.ay[env] = ay; s.avx[env] = avx; s.avy[env] = avy;
            s.next_vx[env] = next_vx; s.next_vy[env] = next_vy; s.input_timer[env] = input_timer;
            s.anim_timer[env] = anim_timer; s.eat_timer[env] = eat_timer; s.anim_index[env] = anim_index;
            c.mti[env] = rng.idx;
            c.sprites_valid[env] = 1;
        }
        *reward = __fadd_rn(__fmul_rn((float)point_delta, 0.04f), __fmul_rn((float)(points_available == 0), 10.0f));
        return dead || points_available == 0;
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV_NOINLINE void regenerate(const State& s, const CommonState& c, int env, WarpCtx& w) {
        const int N = s.N, lane = w.lane;
        uint8_t* tiles = w.alloc<uint8_t>(TILE_STRIDE);   // 0 empty, 1 wall, 2 marker
        uint8_t* kinds = w.alloc<uint8_t>(MAX_ENTS);
        cell_t* cells = w.alloc<cell_t>(MAX_ENTS);
        cell_t* quad = w.alloc<cell_t>(4 * QUAD_CAP);
        cell_t* fc = w.alloc<cell_t>(FC_CAP);
        uint8_t* order = w.alloc<uint8_t>(MAX_ENTS);
        Set* us = w.alloc<Set>(1);
        int nents = 0;

        MazeGrid mg = kruskal_maze(w, W, H);
        const int extra_quad = w.rng.uniform_int(0, 3);   // drawn in every mode (extra_orb_sign == 0 in easy mode)

        int nq[4] = { 0, 0, 0, 0 };
        for (int x = 0; x < W; x++)
            for (int y = 0; y < H; y++) {
                int obj = mg.get(x + 1, y + 1);
                tiles[y + x * H] = obj == 1 ? 1 : 0;
                if (obj == 0) {
                    int qi = (x >= W / 2) * 2 + (y >= H / 2);
                    if (nq[qi] < QUAD_CAP) quad[qi * QUAD_CAP + nq[qi]] = (cell_t)(y + x * H);
                    nq[qi]++;
                }
            }
        __syncwarp();
        bool quad_overflow = false;
        for (int i = 0; i < 4; i++) {
            // 1 + (i == extra_quad ? extra_orb_sign : 0) orbs per quadrant, distinct positions, spawned in the
            // iteration order of the local unordered_set (tilemap.cpp:146-170)
            if (nq[i] > QUAD_CAP) { quad_overflow = true; nq[i] = QUAD_CAP; }
            const int num_orbs = 1 + (i == extra_quad ? ORB_SIGN : 0);
            us->init(1);
            for (int j = 0; j < num_orbs; j++) {
                int pos = w.rng.uniform_int(0, nq[i] - 1);
                while (us->count > 0 && us->contains(pos)) pos = (pos + 1) % nq[i];
                us->insert(pos);
            }
            const int nsel = us->order(order);
            __syncwarp();
            for (int j = 0; j < nsel; j++) {
                int cell = quad[i * QUAD_CAP + order[j]];
                kinds[nents] = K_ORB; cells[nents] = (cell_t)cell; nents++;
                tiles[cell] = 2;
            }
            __syncwarp();
        }
        int nfree = 0;
        for (int i = 0; i < W * H; i++) if (tiles[i] == 0) { if (nfree < FC_CAP) fc[nfree] = (cell_t)i; nfree++; }
        __syncwarp();
        // agent + 3 eggs: distinct positions into free_cells, walked in unordered_set order (Q4)
        us->init(1);
        for (int j = 0; j < NMOB + 1; j++) {
            int pos = w.rng.uniform_int(0, nfree - 1);
            while (us->count > 0 && us->contains(pos)) pos = (pos + 1) % nfree;
            us->insert(pos);
        }
        int nsel = us->order(order);
        (void)nsel;
        const int start = fc[order[0]];
        const int agent_spawn_x = start / H, agent_spawn_y = start % H;
        int egg_cell[NMOB];
        tiles[start] = 2;
        for (int i = 0; i < NMOB; i++) {
            egg_cell[i] = fc[order[1 + i]];
            kinds[nents] = K_MOB; cells[nents] = (cell_t)egg_cell[i]; nents++;
            tiles[egg_cell[i]] = 2;
        }
        __syncwarp();
        nfree = 0;
        for (int i = 0; i < W * H; i++) if (tiles[i] == 0) { if (nfree < FC_CAP) fc[nfree] = (cell_t)i; nfree++; }
        for (int i = 0; i < nfree && nents < MAX_ENTS; i++) { kinds[nents] = K_POINT; cells[nents] = fc[i]; nents++; }
        __syncwarp();

        // ---- reset() tail (chaser.cpp:425-446)
        int bg_index = w.rng.uniform_int(0, NUM_BG - 1);
        float bg_offset = w.rng.uniform_real(0.0f, 1.0f);

        // ---- ECS set orders: sprite_render = every entity above (ids ascending), mob_ai = eggs (ids NORB ..)
        us->init(s.nb_sprite[env]);
        for (int e = 0; e < nents; e++) us->insert(e);
        int n_sprite = us->order(order);
        int nb_sprite = us->nb;
        __syncwarp();
        for (int k = lane; k < n_sprite; k += WARP_LANES) s.sprite_order[k * N + env] = order[k];
        __syncwarp();
        us->init(s.nb_mob[env]);
        for (int i = 0; i < NMOB; i++) us->insert(NORB + i);
        us->order(order);
        int nb_mob = us->nb;
        __syncwarp();
        for (int k = lane; k < NMOB; k += WARP_LANES) s.mob_order[k * N + env] = (uint8_t)(order[k] - NORB);

        uint8_t* gt = s.tiles + (size_t)env * TILE_STRIDE;
        for (int i = lane; i < W * H; i += WARP_LANES) gt[i] = tiles[i] == 1 ? 1 : 0;   // markers cleared
        cell_t* gf = s.free_cells + (size_t)env * FREE_STRIDE;
        for (int i = lane; i < nfree && i < FREE_STRIDE; i += WARP_LANES) gf[i] = fc[i];
        for (int e = lane; e < nents; e += WARP_LANES) { s.ent_kind[e * N + env] = kinds[e]; s.ent_cell[e * N + env] = cells[e]; }
        for (int i = lane; i < NMOB; i += WARP_LANES) {
            s.mob_x[i * N + env] = __fadd_rn((float)(egg_cell[i] / H), 0.5f);
            s.mob_y[i * N + env] = __fadd_rn((float)(H - 1 - egg_cell[i] % H), 0.5f);
            s.mob_vx[i * N + env] = 0.0f; s.mob_vy[i * N + env] = 0.0f;
            s.mob_hatch[i * N + env] = 0.0f; s.mob_tex[i * N + env] = T_EGG;
        }
        if (lane == 0) {
            s.num_free[env] = nfree;
            s.num_ents[env] = nents;
            s.nb_sprite[env] = nb_sprite; s.nb_mob[env] = nb_mob;
            s.anim_timer[env] = 0.0f; s.anim_index[env] = 0; s.eat_timer[env] = 0.0f;
            s.ax[env] = __fadd_rn((float)agent_spawn_x, 0.5f);
            s.ay[env] = __fadd_rn((float)(H - 1 - agent_spawn_y), 0.5f);
            s.avx[env] = 0.0f; s.avy[env] = 0.0f; s.next_vx[env] = 0.0f; s.next_vy[env] = 0.0f; s.input_timer[env] = 0.0f;
            s.bg_index[env] = bg_index; s.bg_offset[env] = bg_offset;
            c.cam_x[env] = __fmul_rn(__fmul_rn((float)W, 0.5f), UNIT_TO_PIXELS);
            c.cam_y[env] = __fmul_rn(__fmul_rn((float)H, 0.5f), UNIT_TO_PIXELS);
            c.sprites_valid[env] = 0;
            if (nfree > FREE_STRIDE || nfree + NORB + NMOB > MAX_ENTS || quad_overflow) c.fault[env] |= 1;
        }
    }

    // ---------------------------------------------------------------------------------------
    static PG2_DEV int tile_class(uint32_t) { return 0; }

    template <class F>
    static PG2_DEV_NOINLINE void build_frame(const State& s, const CommonState& c, int env, F& f, const TexInfo* tex) {
        const int N = s.N;
        // game_zoom = width * pixels_to_unit / map_width (chaser.cpp:401)
        Camera cam{ c.cam_x[env], c.cam_y[env], __fdiv_rn(__fmul_rn(f.view_w, PIXELS_TO_UNIT), (float)W), f.view_w, f.view_h };
        int lx, ly, ux, uy;
        tile_window(cam, &lx, &ly, &ux, &uy);
        const int ncol = min(ux - lx + 1, MAX_WIN), nrow = min(uy - ly + 1, MAX_WIN);
        const int nents = s.num_ents[env];
        const bool sprites = c.sprites_valid[env] != 0;
        // background (e.g. maze.cpp:402-408): the blit itself is built by build_tile_layer below
        const int bg = T_BG0 + s.bg_index[env];
        const TexInfo bt = tex[bg];
        const float bg_x = __fmul_rn(-s.bg_offset[env], __fsub_rn(__fdiv_rn((float)bt.w, (float)bt.h), 1.0f));
        const float bg_scale = __fdiv_rn(__fmul_rn(64.0f, UNIT_TO_PIXELS), (float)bt.h);
        const int nlive = live_list(f, sprites ? nents : 0, [&](int j) {
            const int e = s.sprite_order[j * N + env];
            return s.ent_kind[e * N + env] != K_NONE ? e : -1; });
        const uint8_t* tiles = s.tiles + (size_t)env * TILE_STRIDE;
        build_tile_layer(f, cam, tex, 1, lx, ly, ncol, nrow, [](int) { return (int)T_WALL; },
                         [&](int x, int y) { return get(tiles, x, H - 1 - y) == 1 ? (int)T_WALL : (int)NO_TILE; }, bg, bg_x, 0.0f, bg_scale);
        emit_post_blits(f, tex, nlive + 1, [&](int k, BlitReq& b, BlitRot&) {
            if (k < nlive) {
                const int e = f.live[sort_perm(nlive, k)];
                int kind = s.ent_kind[e * N + env];
                int t; float x, y;
                if (kind == K_MOB) {
                    int m = e - NORB;
                    t = s.mob_tex[m * N + env]; x = s.mob_x[m * N + env]; y = s.mob_y[m * N + env];
                } else {
                    int cell = s.ent_cell[e * N + env];
                    t = kind == K_ORB ? T_CRYSTAL : T_POINT;
                    x = __fadd_rn((float)(cell / H), 0.5f); y = __fadd_rn((float)(H - 1 - cell % H), 0.5f);
                }
                float px = __fmul_rn(__fadd_rn(x, -0.5f), UNIT_TO_PIXELS);
                float py = __fmul_rn(__fadd_rn(y, -0.5f), UNIT_TO_PIXELS);
                float sc = __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, 1.0f), UNIT_TO_PIXELS), (float)tex[t].w);
                b.plain(t, px, py, cam, sc);
            } else {
                float px = __fmul_rn(__fadd_rn(s.ax[env], -0.5f), UNIT_TO_PIXELS);
                float py = __fmul_rn(__fadd_rn(s.ay[env], -0.5f), UNIT_TO_PIXELS);
                b.plain(T_AGENT, px, py, cam, __fmul_rn(__fdiv_rn(UNIT_TO_PIXELS, (float)tex[T_AGENT].w), 1.0f));
            }
        });
    }
};
using Chaser = ChaserT<0>;

}  // namespace pg2
