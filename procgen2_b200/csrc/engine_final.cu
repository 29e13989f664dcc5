// k_render<G, true> (pg2_kernels.cuh) for every game; engine.cu launches it through the address render_final_kernel<G>
// returns. A translation unit of its own: the device code of engine.cu, and so every kernel an engine without final_obs
// launches, compiles exactly as it would without these kernels. Its device globals are its own too: the sort table
// pointer is set here as well (ensure_sort_table).
#define PG2_TU_LOCAL static   // see pg2_platform.cuh
#include <cuda_runtime.h>

#include "games/all_games.cuh"
#include "pg2_kernels.cuh"

namespace pg2 {

cudaError_t final_set_sort_table(const uint8_t* table) { return cudaMemcpyToSymbol(g_sort_perm, &table, sizeof(table)); }

template <class G>
const void* render_final_kernel() { return (const void*)k_render<G, true>; }

#define PG2_FINAL_GAME(NAME, TYPE) template const void* render_final_kernel<TYPE>();
#define PG2_FINAL_GAME_MODE(NAME, MODE, TYPE) PG2_FINAL_GAME(NAME, TYPE)
PG2_FOR_EACH_GAME(PG2_FINAL_GAME)
PG2_FOR_EACH_GAME_MODE(PG2_FINAL_GAME_MODE)

}  // namespace pg2
