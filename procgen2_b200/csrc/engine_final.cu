// k_render_final<G> (pg2_kernels.cuh) for every game, and the host calls engine.cu makes to it. A translation unit of its
// own: the device code of engine.cu, and so every kernel an engine without final_obs launches, compiles exactly as it
// would without these kernels. Its device globals are its own too: the sort table pointer is set here as well
// (ensure_sort_table).
#define PG2_TU_LOCAL static   // see pg2_platform.cuh
#include <cuda_runtime.h>

#include "games/all_games.cuh"
#include "pg2_kernels.cuh"

namespace pg2 {

cudaError_t final_set_sort_table(const uint8_t* table) { return cudaMemcpyToSymbol(g_sort_perm, &table, sizeof(table)); }

template <class G>
cudaError_t render_final_occupancy(int* ctas_per_sm) {
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, k_render_final<G>, RENDER_THREADS, 0);
}

template <class G>
void launch_render_final(int grid, cudaStream_t on, const typename G::State& s, const CommonState& c, const TexInfo* tex, const uint32_t* atlas,
                         uint8_t* obs, int* ticket, int mode, const int* list, const int* list_count, const uint8_t* pending, int N,
                         uint8_t* view_cache, const SwapArgs& swap, uint8_t* final_obs, int* zero_ticket) {
    k_render_final<G><<<grid, RENDER_THREADS, 0, on>>>(s, c, tex, atlas, obs, ticket, mode, list, list_count, pending, N, view_cache, swap,
                                                       final_obs, zero_ticket);
}

#define PG2_FINAL_INSTANTIATE(TYPE)                                                                                              \
    template cudaError_t render_final_occupancy<TYPE>(int*);                                                                     \
    template void launch_render_final<TYPE>(int, cudaStream_t, const TYPE::State&, const CommonState&, const TexInfo*, const uint32_t*, \
                                            uint8_t*, int*, int, const int*, const int*, const uint8_t*, int, uint8_t*, const SwapArgs&, \
                                            uint8_t*, int*);
#define PG2_FINAL_GAME(NAME, TYPE) PG2_FINAL_INSTANTIATE(TYPE)
#define PG2_FINAL_GAME_MODE(NAME, MODE, TYPE) PG2_FINAL_INSTANTIATE(TYPE)
PG2_FOR_EACH_GAME(PG2_FINAL_GAME)
PG2_FOR_EACH_GAME_MODE(PG2_FINAL_GAME_MODE)

}  // namespace pg2
