// Randomised-Kruskal maze generator shared by maze, chaser and jumper.
// Reference: Maze_Generator::generate_maze — games/maze/maze_generator.cpp:55-139 (union-find with path
// halving / union by rank) and games/chaser/maze_generator.cpp:47-130 == games/jumper/maze_generator.cpp
// (per-cell unordered_set merging). Both consume the RNG identically — one uniform_int(0, walls-1) per
// wall, wall list built in the same order, walls.erase(begin + n) — and produce identical grids
// (SURVEY Q6), so ONE device union-find generator serves all three games.
// One warp, redundant-uniform execution (pg2_warp.cuh); only the wall-list erase is lane-parallel.
#pragma once
#include "pg2_warp.cuh"

namespace pg2 {

constexpr int MAZE_MAX_DIM = 31;                                   // maze_dim <= 31 (maze memory mode)
constexpr int MAZE_MAX_ARR = (MAZE_MAX_DIM + 2) * (MAZE_MAX_DIM + 2);

struct MazeGrid {
    int mw, mh, aw, ah;        // maze size, padded array size
    uint8_t* grid;             // [y + ah * x], 1 wall / 0 space (/ 2 object), padded by one cell
    int16_t* free_cells;       // cell indices (y + mh * x) in the order they were freed
    int num_free;
    PG2_DEV int get(int x, int y) const {                          // Maze_Generator::get (padded coords)
        if (x < 0 || y < 0 || x >= aw || y >= ah) return 1;
        return grid[y + ah * x];
    }
};

PG2_TU_LOCAL PG2_DEV_NOINLINE MazeGrid kruskal_maze(WarpCtx& w, int mw, int mh) {
    const int lane = w.lane;
    MazeGrid m;
    m.mw = mw; m.mh = mh; m.aw = mw + 2; m.ah = mh + 2;
    const int ah = m.ah;
    // scratch sized by THIS maze (11x11 chaser ... 31x31 maze memory mode), so every game's arena only pays for its own
    const int arr = m.aw * m.ah, cells = mw * mh;
    m.grid = w.alloc<uint8_t>(arr);
    m.free_cells = w.alloc<int16_t>(arr);
    int16_t* set_idx = w.alloc<int16_t>(arr);
    uint8_t* set_rank = w.alloc<uint8_t>(arr);
    uint8_t* is_free = w.alloc<uint8_t>(cells);
    uint32_t* walls = w.alloc<uint32_t>(cells / 2 + 4);             // x1 | y1<<8 | x2<<16 | y2<<24 (31x31: 480 walls)
    uint8_t* grid = m.grid;
    int16_t* free_cells = m.free_cells;
    w.fill<uint8_t>(grid, m.aw * m.ah, 1);
    w.fill<uint8_t>(is_free, cells, 0);
    for (int i = lane; i < mw * mh; i += WARP_LANES) { set_idx[i] = (int16_t)i; set_rank[i] = 0; }
    __syncwarp();
    grid[1 + ah * 1] = 0;                                          // corner
    int num_free = 0;
    int nwalls = 0;
    for (int i = 1; i < mw; i += 2)
        for (int j = 0; j < mh; j += 2)
            if (i > 0 && i < mw - 1) { walls[nwalls] = (uint32_t)(i - 1) | (uint32_t)j << 8 | (uint32_t)(i + 1) << 16 | (uint32_t)j << 24; nwalls++; }
    for (int i = 0; i < mw; i += 2)
        for (int j = 1; j < mh; j += 2)
            if (j > 0 && j < mh - 1) { walls[nwalls] = (uint32_t)i | (uint32_t)(j - 1) << 8 | (uint32_t)i << 16 | (uint32_t)(j + 1) << 24; nwalls++; }
    __syncwarp();

    auto find = [&](int cell) {                                    // path halving
        int cur = cell;
        while (set_idx[cur] != cur) { int gp = set_idx[set_idx[cur]]; set_idx[cur] = (int16_t)gp; cur = gp; }
        return cur;
    };
    auto set_free_cell = [&](int x, int y) {
        grid[(y + 1) + ah * (x + 1)] = 0;
        int cell = y + mh * x;
        if (!is_free[cell]) { free_cells[num_free] = (int16_t)cell; is_free[cell] = 1; num_free++; }
    };

    while (nwalls > 0) {
        int n = w.rng.uniform_int(0, nwalls - 1);
        uint32_t wl = walls[n];
        int x1 = wl & 255, y1 = (wl >> 8) & 255, x2 = (wl >> 16) & 255, y2 = wl >> 24;
        int s0 = find(y1 + mh * x1);
        int s1 = find(y2 + mh * x2);
        int x0 = (x1 + x2) / 2, y0 = (y1 + y2) / 2;
        int center = y0 + mh * x0;
        bool can_remove = (grid[(y0 + 1) + ah * (x0 + 1)] == 1) && (s0 != s1);
        __syncwarp();
        if (can_remove) {
            set_free_cell(x1, y1);
            set_free_cell(x0, y0);
            set_free_cell(x2, y2);
            if (set_rank[s0] > set_rank[s1]) {
                set_idx[s1] = (int16_t)s0; set_idx[center] = (int16_t)s0;
            } else {
                set_idx[s0] = (int16_t)s1; set_idx[center] = (int16_t)s1;
                if (set_rank[s0] == set_rank[s1]) set_rank[s1]++;
            }
        }
        __syncwarp();
        // walls.erase(walls.begin() + n): order-preserving shift, 32 elements at a time
        for (int base = n; base < nwalls - 1; base += WARP_LANES) {
            int k = base + lane;
            uint32_t v = (k < nwalls - 1) ? walls[k + 1] : 0u;
            __syncwarp();
            if (k < nwalls - 1) walls[k] = v;
            __syncwarp();
        }
        nwalls--;
    }
    m.num_free = num_free;
    return m;
}

}  // namespace pg2
