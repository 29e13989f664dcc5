// Maze — device restatement of /root/reference/games/maze/:
//   step logic   System_Agent::update          common_systems.cpp:69-136, cenv_step maze.cpp:279-326
//   level gen    System_Tilemap::regenerate    tilemap.cpp:31-109, Maze_Generator maze_generator.cpp:47-195,
//                reset()                       maze.cpp:416-438
//   frame        render_game                   maze.cpp:386-414, tilemap.cpp:111-131,
//                sprite / agent render         common_systems.cpp:41-63, 138-151
// All three distribution modes of tilemap.cpp:35-47 as MazeT<MODE> (0 easy: 15x15 world; 1 hard, the reference's compiled-in
// default: 25x25; 2 memory: 31x31 world, an 8x8-tile view that follows the agent).
#pragma once
#include "../pg2_common.cuh"
#include "../pg2_mazegen.cuh"
#include "../pg2_render.cuh"
#include "../pg2_state.cuh"
#include "../pg2_warp.cuh"

namespace pg2 {

#define PG2_MAZE_FIELDS(F)                                              \
    PG2_ENV_MAJOR(F)(uint8_t, tiles, 1024) /* [y + x*WORLD] (WORLD <= 31), 0 empty 1 wall */ \
    F(float, agent_x, 1)                                                \
    F(float, agent_y, 1)                                                \
    F(uint8_t, face_forward, 1)                                         \
    F(float, goal_x, 1)                                                 \
    F(float, goal_y, 1)                                                 \
    F(int32_t, bg_index, 1)                                             \
    F(float, bg_offset, 1)                                              \
    F(int32_t, curr_step, 1)

PG2_DEFINE_STATE(MazeState, PG2_MAZE_FIELDS)

template <int MODE>
struct MazeT {
    using State = MazeState;
    static constexpr int WORLD = MODE == 1 ? 25 : MODE == 2 ? 31 : 15;     // world_dim (tilemap.cpp:35-47)
    static constexpr int VISIBLE = MODE == 1 ? 25 : MODE == 2 ? 8 : 15;    // visibility: the zoom's denominator (maze.cpp:397)
    static constexpr bool CENTER_AGENT = MODE == 2;                        // memory mode: the camera follows the agent from its first update on
    static constexpr int TIMEOUT = 500;       // maze.cpp:49
    static constexpr bool LANE_AWARE = false;   // step() is written for one thread per environment
    static constexpr int STEP_LANES = 32;       // (lane-aware games only) lanes per environment in k_step
    static constexpr int MAX_POST = 4;        // capacity of the frame's post-blit list
    static constexpr bool ROTATES = false;     // some blits are rotated
    static constexpr bool SLOW_RESET = true;   // level generation is long: run it concurrently with the render of the other envs
    static constexpr int RESET_ARENA = 13 * 1024;   // per-warp level-generation scratch (high water measured with PG2_ARENA_TRACE; 31x31 mazes)
    static constexpr bool PREFETCH_LEVELS = true;    // the RNG is only drawn inside reset(): the next level is generated one episode ahead
    static constexpr int PREFETCH_MIN_EPISODE = 0;   // level prefetch whatever max_episode_steps is
    static const char* reset_keeps() { return "  "; }   // fields reset() does not write (they persist across episodes)
    static constexpr int TILE_CLASSES = 1;
    static constexpr int WIN_ROWS = 28;        // most tile rows the camera window can span (zoom-dependent; frame table sizing)
    static constexpr int BLIT_UNROLL = 1;     // post-blit patches fetched together (pg2_render.cuh draw_blit_band)
    static constexpr int RENDER_MIN_CTAS = 7;   // CTAs per SM the register allocation of k_render aims at
    static constexpr int DEFAULT_MODE = MODE;    // this instantiation's distribution mode (the reference compiles in 1 = hard; tilemap.h Config)
    static bool mode_supported(int mode) { return mode == MODE; }
    static constexpr bool HAS_TILES = true;     // the frame has a tile layer
    static constexpr bool STATIC_VIEW = !CENTER_AGENT;   // fixed camera and tile map within an episode: the base image (background + tiles) is cached per env
    static constexpr int TILE_STRIDE = 1024;
    enum Tex { T_WALL = 0, T_CHEESE = 1, T_MOUSE = 2, T_BG0 = 3, NUM_BG = 9, NUM_TEX = 12 };

    static const char* const* texture_names(int* count) {
        static const char* const names[NUM_TEX] = {
            "assets/kenney/Ground/Sand/sandCenter.png",
            "assets/misc_assets/cheese.png",
            "assets/kenney/Enemies/mouse_move.png",
            "assets/topdown_backgrounds/floortiles.png",
            "assets/topdown_backgrounds/backgrounddetailed1.png",
            "assets/topdown_backgrounds/backgrounddetailed2.png",
            "assets/topdown_backgrounds/backgrounddetailed3.png",
            "assets/topdown_backgrounds/backgrounddetailed4.png",
            "assets/topdown_backgrounds/backgrounddetailed5.png",
            "assets/topdown_backgrounds/backgrounddetailed6.png",
            "assets/topdown_backgrounds/backgrounddetailed7.png",
            "assets/topdown_backgrounds/backgrounddetailed8.png",
        };
        *count = NUM_TEX;
        return names;
    }

    // System_Tilemap::get (tilemap.h:79-84): out of bounds is a wall. (x, y) in map space.
    static PG2_DEV int get(const uint8_t* tiles, int x, int y) {
        if (x < 0 || y < 0 || x >= WORLD || y >= WORLD) return 1;
        return tiles[y + x * WORLD];
    }

    // ---------------------------------------------------------------------------------------
    // cenv_step body for one environment (thread-per-env). Returns terminated.
    static PG2_DEV_NOINLINE bool step(const State& s, const CommonState& c, int env, int action, float* reward, const StepCtx& ctx) {
        const uint8_t* tiles = s.tiles + (size_t)env * TILE_STRIDE;
        float px = s.agent_x[env], py = s.agent_y[env];
        int movement_x = action / 3 - 1;
        int movement_y = movement_x ? 0 : -(action % 3 - 1);
        if (movement_x) {
            int nx = f2i(__fadd_rn(px, (float)movement_x));
            if (get(tiles, nx, WORLD - 1 - f2i(py)) == 0) px = __fadd_rn((float)nx, 0.5f);
        } else if (movement_y) {
            int ny = f2i(__fadd_rn(py, (float)movement_y));
            if (get(tiles, f2i(px), WORLD - 1 - ny) == 0) py = __fadd_rn((float)ny, 0.5f);
        }
        Rect me{ __fadd_rn(px, -0.5f), __fadd_rn(py, -0.5f), 1.0f, 1.0f };
        Rect goal{ __fadd_rn(s.goal_x[env], -0.5f), __fadd_rn(s.goal_y[env], -0.5f), 1.0f, 1.0f };
        bool reached = check_collision(me, goal);
        if (movement_x > 0) s.face_forward[env] = 1;
        else if (movement_x < 0) s.face_forward[env] = 0;
        s.agent_x[env] = px; s.agent_y[env] = py;
        if (CENTER_AGENT) {                       // camera follows the agent (common_systems.cpp:119-123: tilemap->center_agent())
            c.cam_x[env] = __fmul_rn(px, UNIT_TO_PIXELS);
            c.cam_y[env] = __fmul_rn(py, UNIT_TO_PIXELS);
        }
        c.sprites_valid[env] = 1;                 // sprite_render->update(dt)
        *reward = reached ? 10.0f : 0.0f;
        bool terminated = reached;
        int cs = s.curr_step[env] + 1;
        s.curr_step[env] = cs;
        if (cs >= TIMEOUT) terminated = true;     // maze.cpp:308-310
        return terminated;
    }

    // ---------------------------------------------------------------------------------------
    // reset(): one warp, redundant-uniform execution (pg2_warp.cuh).
    static PG2_DEV_NOINLINE void regenerate(const State& s, const CommonState& c, int env, WarpCtx& w) {
        const int lane = w.lane;
        uint8_t* tiles = w.alloc<uint8_t>(TILE_STRIDE);
        w.fill<uint8_t>(tiles, TILE_STRIDE, 1);                       // std::fill(..., wall)

        const int maze_dim = w.rng.uniform_int(0, (WORLD - 1) / 2 - 1) * 2 + 3;
        const int margin = (WORLD - maze_dim) / 2;

        // ---- Maze_Generator::generate_maze(maze_dim, maze_dim) (maze_generator.cpp:55-139)
        MazeGrid mg = kruskal_maze(w, maze_dim, maze_dim);
        const int mh = mg.mh, ah = mg.ah, num_free = mg.num_free;
        uint8_t* grid = mg.grid;
        const int16_t* free_cells = mg.free_cells;

        // ---- place_object(GOAL) (maze_generator.cpp:183-195): cell index 10 (START_CELL) and
        // consumed cells are rejected and redrawn (SURVEY Q27)
        int fidx = w.rng.uniform_int(0, num_free - 1);
        while (free_cells[fidx] == -1 || free_cells[fidx] == 10) fidx = w.rng.uniform_int(0, num_free - 1);
        int obj_cell = free_cells[fidx];
        __syncwarp();
        grid[(obj_cell % mh + 1) + ah * (obj_cell / mh + 1)] = 2;
        __syncwarp();

        // ---- copy the maze into the world (tilemap.cpp:77-88)
        int goal_x = 0, goal_y = 0;
        for (int i = 0; i < maze_dim; ++i)
            for (int j = lane; j < maze_dim; j += WARP_LANES) {
                int t = grid[(j + 1) + ah * (i + 1)];
                tiles[(j + margin) + (i + margin) * WORLD] = (t == 1) ? 1 : 0;
            }
        goal_x = obj_cell / mh + margin;
        goal_y = obj_cell % mh + margin;
        __syncwarp();

        // ---- reset() tail (maze.cpp:421-437)
        int bg_index = w.rng.uniform_int(0, NUM_BG - 1);
        float bg_offset = w.rng.uniform_real(0.0f, 1.0f);

        uint8_t* gt = s.tiles + (size_t)env * TILE_STRIDE;
        for (int i = lane; i < TILE_STRIDE / 4; i += WARP_LANES) ((uint32_t*)gt)[i] = ((const uint32_t*)tiles)[i];
        if (lane == 0) {
            s.goal_x[env] = __fadd_rn((float)goal_x, 0.5f);
            s.goal_y[env] = __fadd_rn((float)(WORLD - 1 - goal_y), 0.5f);
            s.agent_x[env] = __fadd_rn((float)margin, 0.5f);
            s.agent_y[env] = __fadd_rn((float)(WORLD - 1 - margin), 0.5f);
            s.face_forward[env] = 1;
            s.bg_index[env] = bg_index;
            s.bg_offset[env] = bg_offset;
            s.curr_step[env] = 0;
            c.cam_x[env] = __fmul_rn(__fmul_rn((float)WORLD, 0.5f), UNIT_TO_PIXELS);
            c.cam_y[env] = __fmul_rn(__fmul_rn((float)WORLD, 0.5f), UNIT_TO_PIXELS);
            c.sprites_valid[env] = 0;
        }
    }

    // ---------------------------------------------------------------------------------------
    // render_game(true): fill the frame description (whole CTA cooperates).
    static PG2_DEV int tile_class(uint32_t) { return 0; }

    template <class F>
    static PG2_DEV_NOINLINE void build_frame(const State& s, const CommonState& c, int env, F& f, const TexInfo* tex) {
        Camera cam{ c.cam_x[env], c.cam_y[env], __fdiv_rn(f.view_w, __fmul_rn(UNIT_TO_PIXELS, (float)VISIBLE)), f.view_w, f.view_h };   // maze.cpp:403: zoom from the width
        int lx, ly, ux, uy;
        tile_window(cam, &lx, &ly, &ux, &uy);
        int ncol = min(ux - lx + 1, MAX_WIN), nrow = min(uy - ly + 1, MAX_WIN);
        // background (e.g. maze.cpp:402-408): the blit itself is built by build_tile_layer below
        const int bg = T_BG0 + s.bg_index[env];
        const TexInfo bt = tex[bg];
        const float bg_x = __fmul_rn(-s.bg_offset[env], __fsub_rn(__fdiv_rn((float)bt.w, (float)bt.h), 1.0f));
        const float bg_scale = __fdiv_rn(__fmul_rn(64.0f, UNIT_TO_PIXELS), (float)bt.h);
        const int ncheese = c.sprites_valid[env] ? 1 : 0;
        // tile layer (tilemap.cpp:111-131)
        const uint8_t* tiles = s.tiles + (size_t)env * TILE_STRIDE;
        build_tile_layer(f, cam, tex, 1, lx, ly, ncol, nrow, [](int) { return (int)T_WALL; },
                         [&](int x, int y) { return get(tiles, x, WORLD - 1 - y) ? (int)T_WALL : (int)NO_TILE; }, bg, bg_x, 0.0f, bg_scale);
        emit_post_blits(f, tex, ncheese + 1, [&](int k, BlitReq& b, BlitRot&) {
            if (k < ncheese) {   // cheese (tilemap.cpp:95-98, common_systems.cpp:41-63)
                float gx = __fmul_rn(__fadd_rn(s.goal_x[env], -0.48f), UNIT_TO_PIXELS);
                float gy = __fmul_rn(__fadd_rn(s.goal_y[env], -0.5f), UNIT_TO_PIXELS);
                float sc = __fdiv_rn(__fmul_rn(__fmul_rn(1.0f, 0.95f), UNIT_TO_PIXELS), (float)tex[T_CHEESE].w);
                b.plain(T_CHEESE, gx, gy, cam, sc);
            } else {             // agent (common_systems.cpp:138-151)
                float ax = __fmul_rn(__fadd_rn(s.agent_x[env], -0.5f), UNIT_TO_PIXELS);
                float ay = __fmul_rn(__fadd_rn(s.agent_y[env], -0.5f), UNIT_TO_PIXELS);
                float sc = __fmul_rn(__fdiv_rn(UNIT_TO_PIXELS, (float)tex[T_MOUSE].w), 1.0f);
                b.plain(T_MOUSE, ax, ay, cam, sc, 1.0f, s.face_forward[env] != 0);
            }
        });
    }
};

using Maze = MazeT<1>;   // the reference's compiled-in mode

}  // namespace pg2
