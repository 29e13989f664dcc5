// Host side of the batched engine + kernel entry points (sm_100a).
//
// Per step, per game G, three kernels run back to back on one stream:
//   k_step<G>    thread-per-env: action decode, sub-step loop (entity update, physics, tile /
//                entity collision), reward / terminated, append finished envs to the reset list
//                (warp ballot + one atomic per warp)                 <- cenv_step  (<g>.cpp)
//   k_reset<G>   warp-per-finished-env: reset() with on-device procedural level generation,
//                continuing the env's MT19937 stream                <- reset()     (<g>.cpp)
//   k_render<G>  CTA-per-env: 64x64x3 observation, TMA bulk store    <- render_game (<g>.cpp) + SDL
// (final_obs engines draw the terminal frames of finished envs too: k_render<G, true>, engine_final.cu, see enqueue_step)
// No CPU fallback exists: every entry point fails loudly when CUDA is unavailable.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/pg2_engine.h"
#include "assets.h"
#include "sort_perm.h"
#include "games/all_games.cuh"
#include "pg2_kernels.cuh"

namespace pg2 {

static thread_local std::string g_error;
static int fail(const std::string& msg) { g_error = msg; return 1; }

#define PG2_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t err__ = (call);                                                             \
        if (err__ != cudaSuccess) {                                                             \
            g_error = std::string(#call) + ": " + cudaGetErrorString(err__);                    \
            return 1;                                                                           \
        }                                                                                       \
    } while (0)

// Every C ABI entry point runs on the engine's device and leaves the caller's current device untouched (a torch / CUDA
// host framework keeps allocating and launching where it was).
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != device) ok = cudaSetDevice(device) == cudaSuccess; else prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define PG2_ON_DEVICE(dev)                                                   \
    DeviceGuard guard__(dev);                                                \
    if (!guard__.ok) return fail("cudaSetDevice failed for the engine's device")

// ------------------------------------------------------------------------------------------------
// kernels

// rng.seed(seed) for envs [0, N) (or the listed ones): seeds[i] given, else base + first + i.
__global__ void k_seed(CommonState c, int N, uint32_t base_seed, const int32_t* __restrict__ seeds, int init_persistent) {
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= N) return;
    seed_body(c, env, seeds ? (uint32_t)seeds[env] : base_seed + (uint32_t)env, init_persistent != 0);
}

// k_step, lane 0 of the warp / lane group that finished an env: wait until the generator has delivered the level this env is
// about to take (ready <=> gen_done >= used; almost always true on arrival — the generator had a whole episode; the poll is
// bounded so that a logic error can never hang the GPU: fault bit 4 instead). The wait sits in k_step, whose CTAs come and
// go, never in the persistent render CTAs, which would keep the generator off the SMs.
__device__ __forceinline__ void swap_wait(const SwapArgs& a, const CommonState& live_c, int env) {
    const int need = a.used[env];
    const volatile int* g = a.gen_done + env;
    int spins = 0;
    while (*g < need && spins < (1 << 18)) { __nanosleep(200); spins++; }
    if (*g < need) live_c.fault[env] |= 4;
    __threadfence();
}

// Finished envs are appended to `list` (ballot + one atomic per warp on *count) and flagged in `pending` (an overlapped
// render skips them). The kernel also zeroes *zero_a / zero_b[0..1]: the list counter the NEXT step appends to (that step's
// consumer of the old value has finished by stream order) and the render's frame tickets.
//
// `epw` = environments per warp (power of two, 1..32): lanes [0, epw) of every warp own one environment each.
// Lane-aware games use epw = 1 (a whole warp per environment, per-entity loops strided over the lanes); the others
// pack several environments into a warp once the batch is large.
template <class G>
__global__ void __launch_bounds__(128) k_step(typename G::State s, CommonState c, const int32_t* __restrict__ actions,
                                              float* __restrict__ reward, uint8_t* __restrict__ terminated,
                                              uint8_t* __restrict__ truncated, int* __restrict__ list, int* __restrict__ count,
                                              uint8_t* __restrict__ pending, int* __restrict__ zero_a, int* __restrict__ zero_b,
                                              int N, int max_episode_steps, int auto_reset, int epw, const __grid_constant__ SwapArgs swap) {
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = gtid & 31;
    if (gtid == 0) { *zero_a = 0; zero_b[0] = 0; zero_b[1] = 0; }
    bool done = false;
    int env;
    if (epw == 1 && G::LANE_AWARE && G::STEP_LANES < 32) {   // a lane group per environment, 32 / STEP_LANES environments per warp
        constexpr int L = G::STEP_LANES;
        env = gtid / L;
        const int gl = lane % L;
        const uint32_t gmask = (L >= 32 ? 0xffffffffu : ((1u << L) - 1u)) << (lane / L * L);
        if (env < N) {
            done = step_body<G>(s, c, env, actions[env], reward, terminated, truncated, max_episode_steps, StepCtx{ gl, L, gmask }) && auto_reset && gl == 0;
            if (gl == 0) pending[env] = done;
        }
    } else if (epw == 1) {   // a whole warp per environment (warp-uniform branch)
        env = gtid >> 5;
        if (env < N) {
            done = step_body<G>(s, c, env, actions[env], reward, terminated, truncated, max_episode_steps, StepCtx{ lane, 32 }) && auto_reset && lane == 0;
            if (lane == 0) pending[env] = done;
        }
    } else {
        env = (gtid >> 5) * epw + lane;
        if (lane < epw && env < N) {
            done = step_body<G>(s, c, env, actions[env], reward, terminated, truncated, max_episode_steps, StepCtx{ 0, 1 }) && auto_reset;
            pending[env] = done;
        }
    }
    unsigned m = __ballot_sync(0xffffffffu, done);
    if (m) {
        int base = 0;
        if (lane == 0) base = atomicAdd(count, __popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (done) list[base + __popc(m & ((1u << lane) - 1u))] = env;
        if (swap.table.n > 0 && done) swap_wait(swap, c, env);   // level prefetch: the env's next level exists (k_render copies it in)
    }
}

// reset_list == nullptr: every env resets (cenv_make / cenv_reset).
template <class G>
__global__ void __launch_bounds__(32 * RESET_WARPS_PER_CTA) k_reset(typename G::State s, CommonState c,
                                                                    const int* __restrict__ reset_list,
                                                                    const int* __restrict__ reset_count, int N,
                                                                    int* __restrict__ gen_done = nullptr) {
    extern __shared__ __align__(16) char smem[];
    const int warp_in_cta = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* mt = (uint32_t*)smem + warp_in_cta * MT_N;
    char* arena = smem + RESET_WARPS_PER_CTA * MT_N * 4 + warp_in_cta * G::RESET_ARENA;
    const int count = reset_list ? *reset_count : N;
    const int total_warps = gridDim.x * RESET_WARPS_PER_CTA;
    for (int w = blockIdx.x * RESET_WARPS_PER_CTA + warp_in_cta; w < count; w += total_warps) {
        int env = reset_list ? reset_list[w] : w;
        reset_body<G>(s, c, env, mt, arena, lane);
        if (gen_done != nullptr) {   // level prefetch: publish "the next level of env exists" (swap_wait polls it)
            __threadfence();
            __syncwarp();
            if (lane == 0) atomicAdd(&gen_done[env], 1);
        }
    }
}

// engine_final.cu. This unit never names k_render<G, true>: instantiating it here, even by taking its address, changes
// the code of every k_render<G, false>.
cudaError_t final_set_sort_table(const uint8_t* table);
template <class G>
const void* render_final_kernel();   // k_render<G, true>

// ------------------------------------------------------------------------------------------------
// host engine

// The std::sort permutation table (pg2_render.cuh: g_sort_perm) is a constant of the process: uploaded once per device by
// the first engine created there, shared by every engine and every lib<Game>.so of the process, never rewritten and never
// freed (16.5 KB) — so no engine can pull it from under another one's kernels.
static int ensure_sort_table(int device) {
    static std::mutex mu;
    static bool done[64] = {};
    std::lock_guard<std::mutex> lock(mu);
    if (device < 0 || device >= 64) return fail("device ordinal out of range");
    if (done[device]) return 0;
    std::vector<uint8_t> table = build_sort_perm(SORT_MAXN);
    uint8_t* dev_table = nullptr;
    PG2_CUDA(cudaMalloc(&dev_table, table.size()));
    PG2_CUDA(cudaMemcpy(dev_table, table.data(), table.size(), cudaMemcpyHostToDevice));
    const uint8_t* p = dev_table;
    PG2_CUDA(cudaMemcpyToSymbol(g_sort_perm, &p, sizeof(p)));
    PG2_CUDA(final_set_sort_table(p));   // the same symbol of engine_final.cu's device code
    PG2_CUDA(cudaDeviceSynchronize());
    done[device] = true;
    return 0;
}

struct EngineBase {
    virtual ~EngineBase() {}
    virtual int reset(const int32_t* seeds) = 0;
    virtual int step_device(const int32_t* actions_dev) = 0;
    virtual int render_human(int env, int width, int height, uint8_t* out_host) = 0;
    virtual bool find_field(const char* name, void** ptr, int* esz, int* pe) = 0;
    virtual size_t state_bytes_per_env() = 0;
    virtual size_t state_alloc_bytes() = 0;     // bytes of state_mem
    virtual uint32_t game_tag() = 0;
    virtual int init_shadow() = 0;              // level prefetch: regenerate every env's next level (after state was written)
    virtual int destroy_graphs() = 0;           // the captured step graphs (they hold pointers into this engine's buffers)

    int device = 0, N = 0, max_episode_steps = 0, auto_reset = 1;
    bool final_on = false;     // pg2_config::final_obs: finished envs' terminal frames go to out[cur].final_obs
    uint32_t base_seed = 0;
    cudaStream_t stream = nullptr;
    int64_t launches = 0;
    int num_sms = 148;
    int step_epw = 1;          // environments per warp in k_step
    int render_ctas_per_sm = 8;   // resident CTAs of k_render per SM (occupancy query)
    int final_ctas_per_sm = 8;    // ... of k_render<G, true> (final_on)
    // device buffers
    void* state_mem = nullptr;
    void* common_mem = nullptr;
    CommonState common;
    // The results of a step. Set 0 is allocated by init and is the only one until pipelined stepping starts; then the
    // steps alternate between the two sets. out[cur] is the set the last step wrote (and the device pointers expose).
    // final_obs (final_on only): row e = the terminal frame of env e, written in the steps in which env e finished.
    struct Outputs { uint8_t* obs = nullptr; float* reward = nullptr; uint8_t* terminated = nullptr; uint8_t* truncated = nullptr;
                     uint8_t* final_obs = nullptr; };
    Outputs out[2];
    int cur = 0;
    int32_t* actions = nullptr;
    int32_t* seeds_dev = nullptr;
    int* reset_list = nullptr;
    int* reset_count = nullptr;      // device counters int[4], see k_step
    int* final_ticket = nullptr;     // final_on without level prefetch: int[2], the terminal-frame pass's ticket by step parity
    uint8_t* pending = nullptr;      // env is in this step's reset list
    int parity = 0;
    bool overlap_reset = false;      // k_reset on a second stream, concurrent with the render of the other envs
    cudaStream_t reset_stream = nullptr;
    cudaEvent_t ev_stepped = nullptr, ev_reset_done = nullptr;
    TexInfo* texinfo = nullptr;
    uint32_t* atlas = nullptr;
    int32_t* actions_pinned = nullptr;
    // depth-1 pipelined stepping (pg2_step_pipelined): output set 1 + a copy stream
    bool pipelined = false;
    int32_t* actions_b[2] = { nullptr, nullptr };
    int32_t* pinned_b[2] = { nullptr, nullptr };
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_step[2] = { nullptr, nullptr }, ev_copy[2] = { nullptr, nullptr }, ev_h2d[2] = { nullptr, nullptr };
    bool copy_pending[2] = { false, false };
    // level prefetch
    bool prefetch = false;
    void* shadow_state_mem = nullptr;
    void* shadow_common_mem = nullptr;
    CommonState shadow_common;
    static constexpr int PREP_SLOTS = 4;   // generator launches that may be in flight (each with a private reset list)
    int* prep_list = nullptr;        // [PREP_SLOTS][N]: private copy of a step's reset list for the asynchronous generator
    int* prep_count = nullptr;       // [PREP_SLOTS]
    int* gen_done = nullptr;         // [N] levels delivered by the generator (beyond the first)
    int* gen_used = nullptr;         // [N] levels taken (swap_copy)
    int prep_slot = 0;
    cudaStream_t prep_streams[4] = { nullptr, nullptr, nullptr, nullptr };   // one per slot: the launches overlap
    cudaEvent_t ev_prepared[PREP_SLOTS] = { nullptr, nullptr, nullptr, nullptr };
    SwapTable swap_table;
    uint8_t* view_cache = nullptr;   // G::STATIC_VIEW: VIEW_CACHE_BYTES per env (k_render keeps the view of an episode)
    // optional per-kernel timing
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;   // 4 per step
    int64_t prof_steps = 0;
    double prof_ms[3] = { 0, 0, 0 };

    // per-step timing marks: 4 on the main stream (k_step | k_reset | rest) + 2 around the main render when it runs
    // on the second stream (overlap_reset)
    std::vector<cudaEvent_t> prof_side;
    int prof_mark() { return prof_mark_to(stream, prof_events); }
    int prof_mark_on(cudaStream_t on) { return prof_mark_to(on, prof_side); }
    int prof_mark_to(cudaStream_t on, std::vector<cudaEvent_t>& v) {
        cudaEvent_t ev;
        if (cudaEventCreate(&ev) != cudaSuccess) return 1;
        cudaEventRecord(ev, on);
        v.push_back(ev);
        return 0;
    }
    int prof_collect() {
        cudaStreamSynchronize(stream);
        if (reset_stream) cudaStreamSynchronize(reset_stream);
        for (size_t i = 0; i + 3 < prof_events.size(); i += 4) {
            for (int k = 0; k < 3; k++) {
                float ms = 0.0f;
                cudaEventElapsedTime(&ms, prof_events[i + k], prof_events[i + k + 1]);
                if (overlap_reset && k == 2) continue;   // exposed wait + tail render: not a kernel time
                prof_ms[k] += ms;
            }
            prof_steps++;
        }
        for (size_t i = 0; i + 1 < prof_side.size(); i += 2) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, prof_side[i], prof_side[i + 1]);
            prof_ms[2] += ms;
        }
        for (auto ev : prof_events) cudaEventDestroy(ev);
        for (auto ev : prof_side) cudaEventDestroy(ev);
        prof_events.clear(); prof_side.clear();
        return 0;
    }

    int alloc_outputs(Outputs& o) {
        PG2_CUDA(cudaMalloc(&o.obs, (size_t)N * OBS_BYTES));
        PG2_CUDA(cudaMalloc(&o.reward, sizeof(float) * N));
        PG2_CUDA(cudaMalloc(&o.terminated, N));
        PG2_CUDA(cudaMalloc(&o.truncated, N));
        if (final_on) {
            PG2_CUDA(cudaMalloc(&o.final_obs, (size_t)N * OBS_BYTES));
            PG2_CUDA(cudaMemsetAsync(o.final_obs, 0, (size_t)N * OBS_BYTES, stream));   // rows are written only when an env finishes
        }
        return 0;
    }

    int free_all() {
        DeviceGuard guard(device);
        if (stream) cudaStreamSynchronize(stream);
        if (pipelined) cudaStreamSynchronize(copy_stream);
        for (Outputs& o : out) { cudaFree(o.obs); cudaFree(o.reward); cudaFree(o.terminated); cudaFree(o.truncated); cudaFree(o.final_obs); }
        cudaFree(final_ticket);
        cudaFree(state_mem); cudaFree(common_mem); cudaFree(actions); cudaFree(seeds_dev); cudaFree(reset_list); cudaFree(reset_count); cudaFree(view_cache);
        for (int j = 0; j < PREP_SLOTS; j++) if (prep_streams[j]) { cudaStreamSynchronize(prep_streams[j]); cudaStreamDestroy(prep_streams[j]); }
        for (int j = 0; j < PREP_SLOTS; j++) if (ev_prepared[j]) cudaEventDestroy(ev_prepared[j]);
        cudaFree(shadow_state_mem); cudaFree(shadow_common_mem); cudaFree(prep_list); cudaFree(prep_count); cudaFree(gen_done); cudaFree(gen_used);
        cudaFree(texinfo); cudaFree(atlas); cudaFree(pending);
        if (reset_stream) { cudaStreamSynchronize(reset_stream); cudaStreamDestroy(reset_stream); cudaEventDestroy(ev_reset_done); }
        if (ev_stepped) cudaEventDestroy(ev_stepped);
        destroy_graphs();
        if (actions_pinned) cudaFreeHost(actions_pinned);
        if (pipelined) {
            for (int k = 0; k < 2; k++) { cudaFree(actions_b[k]); cudaFreeHost(pinned_b[k]); cudaEventDestroy(ev_step[k]); cudaEventDestroy(ev_copy[k]); cudaEventDestroy(ev_h2d[k]); }
            cudaStreamDestroy(copy_stream);
        }
        if (stream) cudaStreamDestroy(stream);
        return 0;
    }
};

template <class G>
struct Engine : EngineBase {
    typename G::State st;
    typename G::State shadow_st;

    int init(const pg2_config* cfg) {
        device = cfg->device; N = cfg->num_envs; max_episode_steps = cfg->max_episode_steps; auto_reset = cfg->auto_reset;
        final_on = cfg->final_obs != 0;
        base_seed = (uint32_t)cfg->seed + (uint32_t)cfg->first_env;
        PG2_CUDA(cudaSetDevice(device));
        cudaDeviceProp prop;
        PG2_CUDA(cudaGetDeviceProperties(&prop, device));
        num_sms = prop.multiProcessorCount;
        PG2_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        // lane-aware games always give a whole warp to an environment; the others pack several environments
        // into a warp once there are >= 8 warps per SM sub-partition
        step_epw = 1;
        if (!G::LANE_AWARE) while (step_epw < 32 && N / (step_epw * 2) >= num_sms * 4 * 8) step_epw *= 2;
        if (const char* o = getenv("PG2_STEP_EPW")) { int v = atoi(o); if (v == 1 || v == 2 || v == 4 || v == 8 || v == 16 || v == 32) step_epw = v; }
        PG2_CUDA(cudaMalloc(&state_mem, G::State::bytes(N)));
        PG2_CUDA(cudaMemsetAsync(state_mem, 0, G::State::bytes(N), stream));
        st = G::State::bind(state_mem, N);
        PG2_CUDA(cudaMalloc(&common_mem, CommonState::bytes(N)));
        PG2_CUDA(cudaMemsetAsync(common_mem, 0, CommonState::bytes(N), stream));
        common = CommonState::bind(common_mem, N);
        if (cfg->distribution_mode >= 0 && !G::mode_supported(cfg->distribution_mode))
            return fail("pg2_create: distribution_mode " + std::to_string(cfg->distribution_mode) + " is not available for this game "
                        "(0 easy, 1 hard, 2 memory / extreme; built: every game's reference default, + easy for coinrun and climber)");
        common.mode = cfg->distribution_mode;
        if (alloc_outputs(out[0])) return 1;
        PG2_CUDA(cudaMemsetAsync(out[0].obs, 0, (size_t)N * OBS_BYTES, stream));
        PG2_CUDA(cudaMemsetAsync(out[0].reward, 0, sizeof(float) * N, stream));
        PG2_CUDA(cudaMemsetAsync(out[0].terminated, 0, N, stream));
        PG2_CUDA(cudaMemsetAsync(out[0].truncated, 0, N, stream));
        PG2_CUDA(cudaMalloc(&actions, sizeof(int32_t) * N));
        PG2_CUDA(cudaMalloc(&seeds_dev, sizeof(int32_t) * N));
        PG2_CUDA(cudaMalloc(&reset_list, sizeof(int) * N));
        if (G::STATIC_VIEW) PG2_CUDA(cudaMalloc(&view_cache, (size_t)N * VIEW_CACHE_BYTES));
        PG2_CUDA(cudaMalloc(&reset_count, 4 * sizeof(int)));
        PG2_CUDA(cudaMemsetAsync(reset_count, 0, 4 * sizeof(int), stream));
        PG2_CUDA(cudaMalloc(&pending, N));
        PG2_CUDA(cudaMemsetAsync(pending, 0, N, stream));
        if (final_on) {
            PG2_CUDA(cudaMalloc(&final_ticket, 2 * sizeof(int)));
            PG2_CUDA(cudaMemsetAsync(final_ticket, 0, 2 * sizeof(int), stream));
        }
        prefetch = G::PREFETCH_LEVELS && auto_reset && !(max_episode_steps > 0 && max_episode_steps < G::PREFETCH_MIN_EPISODE);
        if (const char* o = getenv("PG2_PREFETCH")) prefetch = atoi(o) != 0 && G::PREFETCH_LEVELS && auto_reset;
        if (prefetch) {
            PG2_CUDA(cudaMalloc(&shadow_state_mem, G::State::bytes(N)));
            PG2_CUDA(cudaMalloc(&shadow_common_mem, CommonState::bytes(N)));
            shadow_st = G::State::bind(shadow_state_mem, N);
            shadow_common = CommonState::bind(shadow_common_mem, N);
            shadow_common.mode = common.mode;
            PG2_CUDA(cudaMalloc(&prep_list, sizeof(int) * PREP_SLOTS * (size_t)N));
            PG2_CUDA(cudaMalloc(&prep_count, PREP_SLOTS * sizeof(int)));
            PG2_CUDA(cudaMemsetAsync(prep_count, 0, PREP_SLOTS * sizeof(int), stream));
            PG2_CUDA(cudaMalloc(&gen_done, sizeof(int) * (size_t)N));
            PG2_CUDA(cudaMalloc(&gen_used, sizeof(int) * (size_t)N));
            {   // the generator's few long-running CTAs must get onto the SMs before the render fills them: highest priority
                int lo = 0, hi = 0;
                PG2_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
                for (int j = 0; j < PREP_SLOTS; j++) PG2_CUDA(cudaStreamCreateWithPriority(&prep_streams[j], cudaStreamNonBlocking, hi));
            }
            for (int j = 0; j < PREP_SLOTS; j++) PG2_CUDA(cudaEventCreateWithFlags(&ev_prepared[j], cudaEventDisableTiming));
            if (build_swap_table()) return 1;
        }
        memset(&swap_args, 0, sizeof(swap_args));
        if (prefetch) { swap_args.table = swap_table; swap_args.shadow_c = shadow_common; swap_args.gen_done = gen_done; swap_args.used = gen_used; }
        PG2_CUDA(cudaEventCreateWithFlags(&ev_stepped, cudaEventDisableTiming));
        if (const char* o = getenv("PG2_GRAPH")) use_graph = atoi(o) != 0;
        overlap_reset = G::SLOW_RESET && auto_reset && !prefetch;
        if (const char* o = getenv("PG2_OVERLAP_RESET")) overlap_reset = atoi(o) != 0 && auto_reset && !prefetch;
        if (overlap_reset) {
            PG2_CUDA(cudaStreamCreateWithFlags(&reset_stream, cudaStreamNonBlocking));
            PG2_CUDA(cudaEventCreateWithFlags(&ev_reset_done, cudaEventDisableTiming));
        }
        PG2_CUDA(cudaMallocHost(&actions_pinned, sizeof(int32_t) * N));
        // texture atlas: decode the game's textures from the packed blob, upload once
        int ntex = 0;
        const char* const* names = G::texture_names(&ntex);
        std::vector<TexInfo> infos(ntex);
        std::vector<uint32_t> texels;
        std::string err;
        if (!load_textures(cfg->assets_path, names, ntex, &infos, &texels, &err)) return fail(err);
        PG2_CUDA(cudaMalloc(&texinfo, sizeof(TexInfo) * ntex));
        PG2_CUDA(cudaMalloc(&atlas, sizeof(uint32_t) * texels.size()));
        PG2_CUDA(cudaMemcpyAsync(texinfo, infos.data(), sizeof(TexInfo) * ntex, cudaMemcpyHostToDevice, stream));
        PG2_CUDA(cudaMemcpyAsync(atlas, texels.data(), sizeof(uint32_t) * texels.size(), cudaMemcpyHostToDevice, stream));
        if (ensure_sort_table(device)) return 1;
        PG2_CUDA(cudaStreamSynchronize(stream));
        PG2_CUDA(cudaFuncSetAttribute(k_reset<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, reset_smem()));
        // persistent render grid = exactly the CTAs that are resident at once (registers / shared memory decide)
        PG2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&render_ctas_per_sm, k_render<G, false>, RENDER_THREADS, 0));
        if (render_ctas_per_sm < 1) render_ctas_per_sm = 1;
        if (const char* o = getenv("PG2_RENDER_CTAS_PER_SM")) render_ctas_per_sm = atoi(o) > 0 ? atoi(o) : render_ctas_per_sm;
        if (final_on) {
            PG2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&final_ctas_per_sm, render_final_kernel<G>(), RENDER_THREADS, 0));
            if (final_ctas_per_sm < 1) final_ctas_per_sm = 1;
            if (const char* o = getenv("PG2_RENDER_CTAS_PER_SM")) final_ctas_per_sm = atoi(o) > 0 ? atoi(o) : final_ctas_per_sm;
        }
        // cenv_make: seed, then reset() once (level #1 is generated and never rendered, Q29)
        k_seed<<<(N + 127) / 128, 128, 0, stream>>>(common, N, base_seed, nullptr, 1);
        launches++;
        launch_reset(st, common, nullptr, nullptr, nullptr, stream);
        if (init_shadow()) return 1;
        PG2_CUDA(cudaGetLastError());
        PG2_CUDA(cudaStreamSynchronize(stream));
        return 0;
    }

    // Fields swap_copy copies from the shadow state: every field of the game state and mt / mti / sprites_valid (+ the camera
    // where reset() sets it), except the ones the game lists as persisting across reset() (G::reset_keeps()).
    int build_swap_table() {
        swap_table.n = 0;
        const std::string keeps = G::reset_keeps();
        bool overflow = false;
        auto add = [&](const char* name, void* live_ptr, void* shadow_ptr, int esz, int per_env, bool env_major) {
            if (keeps.find(std::string(" ") + name + " ") != std::string::npos) return;
            if (swap_table.n >= MAX_SWAP_FIELDS) { overflow = true; return; }
            swap_table.f[swap_table.n++] = SwapField{ (char*)live_ptr, (const char*)shadow_ptr, esz, per_env, env_major ? 1 : 0 };
        };
        std::vector<void*> shadow_ptrs;
        shadow_st.for_each_field([&](const char*, void* p, int, int, bool) { shadow_ptrs.push_back(p); });
        size_t i = 0;
        st.for_each_field([&](const char* name, void* p, int esz, int pe, bool em) { add(name, p, shadow_ptrs[i++], esz, pe, em); });
        std::vector<void*> shadow_cptrs;
        shadow_common.for_each_field([&](const char*, void* p, int, int, bool) { shadow_cptrs.push_back(p); });
        i = 0;
        common.for_each_field([&](const char* name, void* p, int esz, int pe, bool em) {
            void* sp = shadow_cptrs[i++];
            if (!strcmp(name, "mt") || !strcmp(name, "mti") || !strcmp(name, "sprites_valid") || !strcmp(name, "cam_x") || !strcmp(name, "cam_y"))
                add(name, p, sp, esz, pe, em);
        });
        if (overflow) return fail("level prefetch: too many state fields for the swap table");
        return 0;
    }

    // Shadow := live, then reset() on the shadow: every env's next level, generated ahead of time. Synchronous (cold path:
    // cenv_make, cenv_reset, pg2_restore, pg2_write_field).
    int init_shadow() override {
        if (!prefetch) return 0;
        for (int j = 0; j < PREP_SLOTS; j++) PG2_CUDA(cudaStreamSynchronize(prep_streams[j]));
        PG2_CUDA(cudaMemcpyAsync(shadow_state_mem, state_mem, G::State::bytes(N), cudaMemcpyDeviceToDevice, stream));
        PG2_CUDA(cudaMemcpyAsync(shadow_common_mem, common_mem, CommonState::bytes(N), cudaMemcpyDeviceToDevice, stream));
        launch_reset(shadow_st, shadow_common, nullptr, nullptr, nullptr, stream);
        PG2_CUDA(cudaMemsetAsync(prep_count, 0, PREP_SLOTS * sizeof(int), stream));
        PG2_CUDA(cudaMemsetAsync(gen_done, 0, sizeof(int) * (size_t)N, stream));   // ready <=> gen_done >= used
        PG2_CUDA(cudaMemsetAsync(gen_used, 0, sizeof(int) * (size_t)N, stream));
        for (int j = 0; j < PREP_SLOTS; j++) PG2_CUDA(cudaEventRecord(ev_prepared[j], stream));
        PG2_CUDA(cudaGetLastError());
        return 0;
    }

    int step_grid() const {
        const int per_warp = (G::LANE_AWARE && step_epw == 1) ? 32 / G::STEP_LANES : step_epw;   // environments per warp
        const int warps = (N + per_warp - 1) / per_warp;
        return (warps * 32 + 127) / 128;
    }
    static int reset_smem() { return RESET_WARPS_PER_CTA * (MT_N * 4 + G::RESET_ARENA); }
    // as many CTAs as fit the SMs' shared memory at once (227 KB per SM, 1 KB reserved per CTA, <= 16): the games with a
    // small level-generation scratch run 8x more resets concurrently than the cave generators
    int reset_grid(int count) const {
        int per_sm = (227 * 1024) / (reset_smem() + 1024);
        per_sm = per_sm > 16 ? 16 : (per_sm < 1 ? 1 : per_sm);
        int ctas = (count + RESET_WARPS_PER_CTA - 1) / RESET_WARPS_PER_CTA;
        return ctas < num_sms * per_sm ? (ctas < 1 ? 1 : ctas) : num_sms * per_sm;
    }
    // One helper per kernel of a step; each enqueues its kernel and counts the launch (pg2_kernel_launches).
    int launch_step(cudaStream_t on) {
        const cudaKernelNodeParams p = step_node_params();
        PG2_CUDA(cudaLaunchKernel(p.func, p.gridDim, p.blockDim, p.kernelParams, p.sharedMemBytes, on));
        launches++;
        return 0;
    }
    // list == nullptr: every env of `s` resets; gen_done: the level generator of the shadow state publishes its levels
    void launch_reset(const typename G::State& s, const CommonState& c, const int* list, const int* count, int* gen_done, cudaStream_t on) {
        k_reset<G><<<reset_grid(N), 32 * RESET_WARPS_PER_CTA, reset_smem(), on>>>(s, c, list, count, N, gen_done);
        launches++;
    }
    // final: a step of a final_on engine. With level prefetch the render of the step draws the terminal frames too (mode 0);
    // without it, final is the pass over the reset list before k_reset (mode 2) that writes the terminal frames.
    int launch_render(int mode, int* ticket, cudaStream_t on, bool final = false) {
        const int per_sm = final ? final_ctas_per_sm : render_ctas_per_sm;
        int grid = N < num_sms * per_sm ? N : num_sms * per_sm;
        // (level prefetch: the list / counter k_step appended this step's finished envs to)
        const int* lst = prefetch && ka_list ? ka_list : reset_list;
        const int* cnt = prefetch && ka_count ? ka_count : reset_count + parity;
        // final with prefetch: reset frames to obs, terminal frames to final_obs; final without: the terminal frames are obs
        uint8_t* obs = final && !prefetch ? out[cur].final_obs : out[cur].obs;
        uint8_t* final_obs = final && prefetch ? out[cur].final_obs : nullptr;
        int* zero_ticket = final && !prefetch ? final_ticket + (parity ^ 1) : nullptr;
        void* args[] = { &st, &common, &texinfo, &atlas, &obs, &ticket, &mode, &lst, &cnt, &pending, &N, &view_cache, &swap_args,
                         &final_obs, &zero_ticket };
        const void* kernel = final ? render_final_kernel<G>() : (const void*)k_render<G, false>;
        PG2_CUDA(cudaLaunchKernel(kernel, dim3(grid), dim3(RENDER_THREADS), args, 0, on));
        launches++;
        return 0;
    }

    int reset(const int32_t* seeds) override {
        if (seeds) {
            // the pinned staging buffer is shared with pg2_step's action copy, which may still be in flight
            PG2_CUDA(cudaStreamSynchronize(stream));
            memcpy(actions_pinned, seeds, sizeof(int32_t) * N);
            PG2_CUDA(cudaMemcpyAsync(seeds_dev, actions_pinned, sizeof(int32_t) * N, cudaMemcpyHostToDevice, stream));
            k_seed<<<(N + 127) / 128, 128, 0, stream>>>(common, N, 0u, seeds_dev, 0);
            launches++;
        }
        launch_reset(st, common, nullptr, nullptr, nullptr, stream);
        if (init_shadow()) return 1;
        PG2_CUDA(cudaMemsetAsync(reset_count + 2, 0, 2 * sizeof(int), stream));
        PG2_CUDA(cudaMemsetAsync(pending, 0, N, stream));   // no env of the last step is waiting for its level swap any more
        ka_list = nullptr; ka_count = nullptr;              // ... and the render below has no swap list (reset_count[0..1] stay zero for these games)
        if (launch_render(0, reset_count + 2, stream)) return 1;
        PG2_CUDA(cudaMemsetAsync(out[cur].reward, 0, sizeof(float) * N, stream));
        PG2_CUDA(cudaMemsetAsync(out[cur].terminated, 0, N, stream));
        PG2_CUDA(cudaMemsetAsync(out[cur].truncated, 0, N, stream));
        PG2_CUDA(cudaGetLastError());
        return 0;
    }

    // ---- one step -------------------------------------------------------------------------------------------------
    // k_step -> k_reset (finished envs) -> k_render on the main stream. Level-prefetch games have no k_reset on that
    // path: finished envs take their pre-generated level in the render CTA that draws them (swap_copy; k_step waits for it to exist), and the level after that is generated on
    // a second stream while the following steps run — up to PREP_SLOTS generator launches in flight, each with a private
    // list (k_step appends to the slot's list directly); an env that finishes again before its next level exists
    // (episodes shorter than a generation) is waited for individually.
    // The main-stream sequence is captured ONCE per (step parity, list slot, output set) into a CUDA graph and
    // replayed: one launch per step; only the pointer to the caller's actions is re-pointed (PG2_GRAPH=0: eager launches).
    // With overlap_reset (PG2_PREFETCH=0 on the slow-generator games) the level generation of the few finished envs runs
    // WHILE a second stream renders all other envs, a short tail render of the reset envs follows (eager only).
    // Timing marks (pg2_profile, eager): [0] k_step, [1] k_reset on the main stream, [2] render (overlap_reset: the
    // render on the second stream; the wait for it and the tail render are not counted).
    // final_on: the terminal frame of a finished env is drawn from the state it finished in, before any reset touches it.
    // With level prefetch that state is still live when the render starts, and the render CTA that swaps the env's level
    // in draws the terminal frame first (k_render<G, true>, no extra launch). Otherwise k_reset overwrites it, so a pass of
    // k_render<G, true> over the reset list runs between k_step and k_reset (one more launch; its time counts as [1]). On the
    // overlap_reset schedule the pass runs before the fork: after it, between the fork and k_reset, it would delay k_reset
    // until the render of the other envs, which fills the SMs meanwhile, has finished (chaser 4096: +55 % per step).
    // The pass's ticket alternates with the step parity: each pass zeroes the one the next step uses.
    SwapArgs swap_args;             // table.n == 0 when the engine does not prefetch levels
    const int32_t* ka_actions = nullptr;
    int *ka_list = nullptr, *ka_count = nullptr, *ka_zero_a = nullptr, *ka_zero_b = nullptr;
    void* step_kargs[16];
    struct StepGraph { cudaGraph_t graph = nullptr; cudaGraphExec_t exec = nullptr; cudaGraphNode_t step_node = nullptr; const int32_t* actions = nullptr;
                       int outputs = -1, kernels = 0; };   // outputs: the output set (out[]) it writes; kernels: its kernel nodes
    StepGraph graphs[2 * PREP_SLOTS];
    bool use_graph = true;

    void bind_step_args(const int32_t* actions_dev, int slot) {
        ka_actions = actions_dev;
        if (prefetch) {
            ka_list = prep_list + (size_t)slot * N; ka_count = prep_count + slot; ka_zero_a = prep_count + (slot + 1) % PREP_SLOTS;
        } else {
            ka_list = reset_list; ka_count = reset_count + parity; ka_zero_a = reset_count + (parity ^ 1);
        }
        ka_zero_b = reset_count + 2;
        Outputs& o = out[cur];
        void* v[16] = { &st, &common, &ka_actions, &o.reward, &o.terminated, &o.truncated, &ka_list, &ka_count, &pending, &ka_zero_a, &ka_zero_b,
                        &N, &max_episode_steps, &auto_reset, &step_epw, &swap_args };
        memcpy(step_kargs, v, sizeof(v));
    }
    cudaKernelNodeParams step_node_params() {
        cudaKernelNodeParams p{};
        p.func = (void*)k_step<G>;
        p.gridDim = dim3(step_grid()); p.blockDim = dim3(128); p.sharedMemBytes = 0;
        p.kernelParams = step_kargs; p.extra = nullptr;
        return p;
    }
    // The main-stream sequence of one step, eager or under stream capture (not overlap_reset).
    int enqueue_step(bool prof) {
        if (prof) prof_mark();
        if (launch_step(stream)) return 1;
        if (prof) prof_mark();
        if (final_on && !prefetch && launch_render(2, final_ticket + parity, stream, true)) return 1;
        if (overlap_reset) {   // fork: the render of all OTHER envs runs on the second stream
            PG2_CUDA(cudaEventRecord(ev_stepped, stream));
            PG2_CUDA(cudaStreamWaitEvent(reset_stream, ev_stepped, 0));
        }
        // (overlap_reset: k_reset stays on the main stream, first in line after k_step, so that its few long-running CTAs
        // get their shared memory before the render fills the SMs)
        if (!prefetch) launch_reset(st, common, reset_list, reset_count + parity, nullptr, stream);
        if (prof) prof_mark();
        if (overlap_reset) {
            if (prof) prof_mark_on(reset_stream);
            if (launch_render(1, reset_count + 2, reset_stream)) return 1;
            if (prof) prof_mark_on(reset_stream);
            PG2_CUDA(cudaEventRecord(ev_reset_done, reset_stream));   // = main render done
            PG2_CUDA(cudaStreamWaitEvent(stream, ev_reset_done, 0));
            if (launch_render(2, reset_count + 3, stream)) return 1;
        } else {
            if (launch_render(0, reset_count + 2, stream, final_on && prefetch)) return 1;
        }
        if (prof) prof_mark();
        return 0;
    }
    int destroy_graphs() override {
        for (auto& g : graphs) if (g.exec) { cudaGraphExecDestroy(g.exec); cudaGraphDestroy(g.graph); g = StepGraph(); }
        return 0;
    }

    int step_device(const int32_t* actions_dev) override {
        parity ^= 1;
        const bool prof = profiling;
        if (prof && prof_events.size() >= 4096) prof_collect();
        const int slot = prep_slot;
        if (prefetch) {
            prep_slot = (prep_slot + 1) % PREP_SLOTS;
            // the generator launches that last read this slot's list / the next slot's counter are done
            PG2_CUDA(cudaStreamWaitEvent(stream, ev_prepared[slot], 0));
            PG2_CUDA(cudaStreamWaitEvent(stream, ev_prepared[(slot + 1) % PREP_SLOTS], 0));
        }
        bind_step_args(actions_dev, slot);
        if (!use_graph || prof || overlap_reset) {
            if (enqueue_step(prof)) return 1;
        } else {
            StepGraph& g = graphs[parity | slot << 1];
            if (g.exec && g.outputs != cur) { cudaGraphExecDestroy(g.exec); cudaGraphDestroy(g.graph); g = StepGraph(); }   // pipelined stepping started
            if (!g.exec) {
                // the capture counts the kernels it records (launch_*): they run in the graph launch below
                cudaGraph_t graph = nullptr;
                PG2_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
                const int rc = enqueue_step(false);
                const cudaError_t ce = cudaStreamEndCapture(stream, &graph);
                if (rc || ce != cudaSuccess || !graph) return fail(std::string("step graph capture failed: ") + cudaGetErrorString(ce));
                size_t nn = 0;
                PG2_CUDA(cudaGraphGetNodes(graph, nullptr, &nn));
                std::vector<cudaGraphNode_t> nodes(nn);
                PG2_CUDA(cudaGraphGetNodes(graph, nodes.data(), &nn));
                for (auto node : nodes) {
                    cudaGraphNodeType ty;
                    cudaKernelNodeParams kp{};
                    if (cudaGraphNodeGetType(node, &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
                    g.kernels++;
                    if (cudaGraphKernelNodeGetParams(node, &kp) == cudaSuccess && kp.func == (void*)k_step<G>) g.step_node = node;
                }
                if (!g.step_node) { cudaGraphDestroy(graph); return fail("step graph: k_step node not found"); }
                PG2_CUDA(cudaGraphInstantiate(&g.exec, graph, 0));
                g.graph = graph;   // kept: the node handle used to re-point `actions` belongs to it
                g.actions = actions_dev; g.outputs = cur;
            } else {
                if (g.actions != actions_dev) {
                    cudaKernelNodeParams kp = step_node_params();
                    PG2_CUDA(cudaGraphExecKernelNodeSetParams(g.exec, g.step_node, &kp));
                    g.actions = actions_dev;
                }
                launches += g.kernels;
            }
            PG2_CUDA(cudaGraphLaunch(g.exec, stream));
        }
        if (prefetch) {
            // the level after the one just taken: generated on the slot's own (high-priority) stream from here on
            PG2_CUDA(cudaEventRecord(ev_stepped, stream));
            PG2_CUDA(cudaStreamWaitEvent(prep_streams[slot], ev_stepped, 0));
            launch_reset(shadow_st, shadow_common, ka_list, ka_count, gen_done, prep_streams[slot]);
            PG2_CUDA(cudaEventRecord(ev_prepared[slot], prep_streams[slot]));
        }
        PG2_CUDA(cudaGetLastError());
        return 0;
    }

    // cenv_render: the env's scene at window resolution (render_game(false)), copied to host memory
    // Blit rects are int16 pixel coordinates (FastBlit), hence at most 32767 pixels per side.
    int render_human(int env, int width, int height, uint8_t* out_host) override {
        if (env < 0 || env >= N || width < 1 || height < 1 || width > 32767 || height > 32767 || (long long)width * height > (1 << 26))
            return fail("pg2_render_human: bad arguments");
        const size_t bytes = (size_t)width * height * 3;
        uint8_t* dev = nullptr;
        PG2_CUDA(cudaMalloc(&dev, bytes + 8));
        int* dev_overflow = (int*)(dev + ((bytes + 3) & ~(size_t)3));
        const int grid = std::max(1, std::min(num_sms * 2, (width * height + 1023) / 1024));
        int overflow = 0;
        cudaError_t ce = cudaMemsetAsync(dev_overflow, 0, sizeof(int), stream);
        if (ce == cudaSuccess) {
            k_render_human<G><<<grid, RENDER_THREADS, 0, stream>>>(st, common, env, texinfo, atlas, dev, width, height, dev_overflow);
            launches++;
            ce = cudaMemcpyAsync(out_host, dev, bytes, cudaMemcpyDeviceToHost, stream);
        }
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(&overflow, dev_overflow, sizeof(int), cudaMemcpyDeviceToHost, stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(stream);
        cudaFree(dev);
        if (ce != cudaSuccess) return fail(std::string("pg2_render_human: ") + cudaGetErrorString(ce));
        if (overflow) return fail("pg2_render_human: the window spans more tile rows than the frame tables hold; use a wider aspect ratio");
        return 0;
    }

    bool find_field(const char* name, void** ptr, int* esz, int* pe) override {
        return st.find(name, ptr, esz, pe) || common.find(name, ptr, esz, pe);
    }
    size_t state_bytes_per_env() override { return (G::State::bytes(1024) + CommonState::bytes(1024)) / 1024; }
    size_t state_alloc_bytes() override { return G::State::bytes(N); }
    uint32_t game_tag() override { return (uint32_t)G::NUM_TEX * 2654435761u ^ (uint32_t)G::State::bytes(1024); }   // distinct per game
};

}  // namespace pg2

// ------------------------------------------------------------------------------------------------
// C ABI

using namespace pg2;

struct pg2_engine { std::unique_ptr<EngineBase> impl; };

extern "C" {

const char* pg2_last_error(void) { return g_error.c_str(); }

int32_t pg2_create(const pg2_config* cfg, pg2_engine** out) {
    if (!cfg || !out || !cfg->game) return fail("pg2_create: null argument");
    if (cfg->num_envs <= 0) return fail("pg2_create: num_envs must be positive");
    if (cfg->final_obs && !cfg->auto_reset)
        return fail("pg2_create: final_obs needs auto_reset = 1 (with auto_reset = 0 the step's observation already is the terminal frame)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail("pg2_create: no CUDA device available — this engine has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= ndev) return fail("pg2_create: invalid device ordinal");
    std::string g = cfg->game;
    for (auto& ch : g) ch = (char)tolower(ch);
    std::unique_ptr<EngineBase> impl;
    int rc = 1;
    PG2_ON_DEVICE(cfg->device);
    // a distribution mode with its own world size is its own instantiation; the others are run-time parameters of the base one
#define PG2_TRY_GAME_MODE(NAME, MODE, TYPE) \
    if (!impl && g == NAME && cfg->distribution_mode == MODE) { auto* e = new Engine<TYPE>(); impl.reset(e); rc = e->init(cfg); }
    PG2_FOR_EACH_GAME_MODE(PG2_TRY_GAME_MODE)
#undef PG2_TRY_GAME_MODE
#define PG2_TRY_GAME(NAME, TYPE) \
    if (!impl && g == NAME) { auto* e = new Engine<TYPE>(); impl.reset(e); rc = e->init(cfg); }
    PG2_FOR_EACH_GAME(PG2_TRY_GAME)
#undef PG2_TRY_GAME
    if (!impl) return fail("pg2_create: unknown game '" + g + "'");
    if (rc) { impl->free_all(); return rc; }
    *out = new pg2_engine{ std::move(impl) };
    return 0;
}

void pg2_destroy(pg2_engine* e) {
    if (!e) return;
    e->impl->free_all();
    delete e;
}

int32_t pg2_reset(pg2_engine* e, const int32_t* seeds) {
    PG2_ON_DEVICE(e->impl->device);
    return e->impl->reset(seeds);
}

int32_t pg2_step(pg2_engine* e, const int32_t* actions_host) {
    EngineBase* b = e->impl.get();
    PG2_ON_DEVICE(b->device);
    // the pinned staging buffer is reused every step: wait for the previous copy to have left it
    PG2_CUDA(cudaStreamSynchronize(b->stream));
    memcpy(b->actions_pinned, actions_host, sizeof(int32_t) * b->N);
    PG2_CUDA(cudaMemcpyAsync(b->actions, b->actions_pinned, sizeof(int32_t) * b->N, cudaMemcpyHostToDevice, b->stream));
    return b->step_device(b->actions);
}

int32_t pg2_render_human(pg2_engine* e, int32_t env, int32_t width, int32_t height, uint8_t* out_rgb) {
    if (!e || !out_rgb) return fail("pg2_render_human: null argument");
    PG2_ON_DEVICE(e->impl->device);
    return e->impl->render_human(env, width, height, out_rgb);
}

int32_t pg2_step_device(pg2_engine* e, const int32_t* actions_device) {
    PG2_ON_DEVICE(e->impl->device);
    return e->impl->step_device(actions_device);
}

// Enqueue the copies of the current results into host buffers (each may be NULL) on `on`.
static int copy_outputs(const EngineBase* b, uint8_t* obs, float* reward, uint8_t* terminated, uint8_t* truncated, cudaStream_t on) {
    const EngineBase::Outputs& o = b->out[b->cur];
    const size_t n = (size_t)b->N;
    if (obs) PG2_CUDA(cudaMemcpyAsync(obs, o.obs, n * OBS_BYTES, cudaMemcpyDeviceToHost, on));
    if (reward) PG2_CUDA(cudaMemcpyAsync(reward, o.reward, sizeof(float) * n, cudaMemcpyDeviceToHost, on));
    if (terminated) PG2_CUDA(cudaMemcpyAsync(terminated, o.terminated, n, cudaMemcpyDeviceToHost, on));
    if (truncated) PG2_CUDA(cudaMemcpyAsync(truncated, o.truncated, n, cudaMemcpyDeviceToHost, on));
    return 0;
}

// pg2_fetch without the wait: the copies are enqueued on the engine's stream (truly asynchronous only into page-locked
// memory, pg2_host_alloc); pg2_sync completes them.
int32_t pg2_fetch_async(pg2_engine* e, uint8_t* obs, float* reward, uint8_t* terminated, uint8_t* truncated) {
    PG2_ON_DEVICE(e->impl->device);
    return copy_outputs(e->impl.get(), obs, reward, terminated, truncated, e->impl->stream);
}

int32_t pg2_fetch(pg2_engine* e, uint8_t* obs, float* reward, uint8_t* terminated, uint8_t* truncated) {
    if (pg2_fetch_async(e, obs, reward, terminated, truncated)) return 1;
    return pg2_sync(e);
}

// Page-locked host memory for result / action buffers (cudaHostAlloc, portable across devices); NULL on failure.
void* pg2_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { g_error = "pg2_host_alloc: cudaHostAlloc failed"; cudaGetLastError(); return nullptr; }
    return p;
}
void pg2_host_free(void* p) { if (p) cudaFreeHost(p); }

// Depth-1 pipelined stepping: enqueue step t (H2D of its actions, the three kernels, D2H of its results into the
// given host buffers on a second stream) and return once the results of step t-1 — written to the buffers passed
// to the PREVIOUS call — are complete. The caller alternates two sets of (pinned) host buffers; outputs are
// double-buffered in HBM so that the copy of step t-1 overlaps the kernels of step t.
static int enable_pipeline(EngineBase* b) {
    const int N = b->N;
    if (b->alloc_outputs(b->out[1])) return 1;
    PG2_CUDA(cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; k++) {
        PG2_CUDA(cudaMalloc(&b->actions_b[k], sizeof(int32_t) * N));
        PG2_CUDA(cudaMallocHost(&b->pinned_b[k], sizeof(int32_t) * N));
        PG2_CUDA(cudaEventCreateWithFlags(&b->ev_step[k], cudaEventDisableTiming));
        PG2_CUDA(cudaEventCreateWithFlags(&b->ev_copy[k], cudaEventDisableTiming));
        PG2_CUDA(cudaEventCreateWithFlags(&b->ev_h2d[k], cudaEventDisableTiming));
    }
    b->pipelined = true;
    return 0;
}

int32_t pg2_step_pipelined(pg2_engine* e, const int32_t* actions_host, uint8_t* obs, float* reward, uint8_t* terminated, uint8_t* truncated) {
    EngineBase* b = e->impl.get();
    PG2_ON_DEVICE(b->device);
    if (!b->pipelined && enable_pipeline(b)) return 1;
    const int prev = b->cur, slot = b->cur ^ 1, N = b->N;
    // this slot's HBM outputs were last read by the copy issued two calls ago, its staging buffer by that call's H2D
    if (b->copy_pending[slot]) PG2_CUDA(cudaStreamWaitEvent(b->stream, b->ev_copy[slot], 0));
    PG2_CUDA(cudaEventSynchronize(b->ev_h2d[slot]));
    memcpy(b->pinned_b[slot], actions_host, sizeof(int32_t) * N);
    PG2_CUDA(cudaMemcpyAsync(b->actions_b[slot], b->pinned_b[slot], sizeof(int32_t) * N, cudaMemcpyHostToDevice, b->stream));
    PG2_CUDA(cudaEventRecord(b->ev_h2d[slot], b->stream));
    b->cur = slot;
    if (b->step_device(b->actions_b[slot])) return 1;
    PG2_CUDA(cudaEventRecord(b->ev_step[slot], b->stream));
    PG2_CUDA(cudaStreamWaitEvent(b->copy_stream, b->ev_step[slot], 0));
    if (copy_outputs(b, obs, reward, terminated, truncated, b->copy_stream)) return 1;
    PG2_CUDA(cudaEventRecord(b->ev_copy[slot], b->copy_stream));
    b->copy_pending[slot] = true;
    if (b->copy_pending[prev]) PG2_CUDA(cudaEventSynchronize(b->ev_copy[prev]));   // results of the previous call are ready
    return 0;
}

// Wait for the results of the last pg2_step_pipelined call.
int32_t pg2_pipeline_flush(pg2_engine* e) {
    EngineBase* b = e->impl.get();
    PG2_ON_DEVICE(b->device);
    if (b->pipelined) PG2_CUDA(cudaStreamSynchronize(b->copy_stream));
    return 0;
}

uint8_t* pg2_obs_device(pg2_engine* e) { return e->impl->out[e->impl->cur].obs; }
float* pg2_reward_device(pg2_engine* e) { return e->impl->out[e->impl->cur].reward; }
uint8_t* pg2_terminated_device(pg2_engine* e) { return e->impl->out[e->impl->cur].terminated; }
uint8_t* pg2_truncated_device(pg2_engine* e) { return e->impl->out[e->impl->cur].truncated; }
uint8_t* pg2_final_obs_device(pg2_engine* e) { return e->impl->out[e->impl->cur].final_obs; }

int32_t pg2_fetch_final_async(pg2_engine* e, const uint8_t* rows, uint8_t* host) {
    const EngineBase* b = e->impl.get();
    if (!b->final_on) return fail("pg2_fetch_final: the engine was created without final_obs");
    if (!host) return fail("pg2_fetch_final: null argument");
    PG2_ON_DEVICE(b->device);
    const uint8_t* src = b->out[b->cur].final_obs;
    for (int i = 0; i < b->N;) {
        if (rows && !rows[i]) { i++; continue; }
        int j = i + 1;
        while (j < b->N && (!rows || rows[j])) j++;
        const size_t off = (size_t)i * OBS_BYTES;
        PG2_CUDA(cudaMemcpyAsync(host + off, src + off, (size_t)(j - i) * OBS_BYTES, cudaMemcpyDeviceToHost, b->stream));
        i = j;
    }
    return 0;
}

int32_t pg2_fetch_final(pg2_engine* e, uint8_t* host) {
    if (pg2_fetch_final_async(e, nullptr, host)) return 1;
    return pg2_sync(e);
}

int32_t pg2_sync(pg2_engine* e) {
    PG2_ON_DEVICE(e->impl->device);
    PG2_CUDA(cudaStreamSynchronize(e->impl->stream));
    return 0;
}
void* pg2_stream(pg2_engine* e) { return (void*)e->impl->stream; }
int32_t pg2_num_envs(pg2_engine* e) { return e->impl->N; }
// Debug builds only (-DPG2_PHASE_TIMERS): reads and clears the render phase counters (pg2_kernels.cuh); -1 otherwise.
int32_t pg2_debug_phases(pg2_engine* e, uint64_t out[8]) {
#ifdef PG2_PHASE_TIMERS
    PG2_ON_DEVICE(e->impl->device);
    unsigned long long z[8] = {};
    PG2_CUDA(cudaDeviceSynchronize());
    PG2_CUDA(cudaMemcpyFromSymbol(out, g_phase, sizeof(z)));
    PG2_CUDA(cudaMemcpyToSymbol(g_phase, z, sizeof(z)));
    return 0;
#else
    (void)e; (void)out;
    return -1;
#endif
}
int32_t pg2_step_epw(pg2_engine* e) { return e->impl->step_epw; }
int64_t pg2_kernel_launches(pg2_engine* e) { return e->impl->launches; }
int64_t pg2_state_bytes_per_env(pg2_engine* e) { return (int64_t)e->impl->state_bytes_per_env(); }

int32_t pg2_profile(pg2_engine* e, int32_t enable) {
    EngineBase* b = e->impl.get();
    DeviceGuard guard__(b->device);
    b->prof_collect();
    b->profiling = enable != 0;
    b->prof_steps = 0;
    b->prof_ms[0] = b->prof_ms[1] = b->prof_ms[2] = 0.0;
    return 0;
}
int32_t pg2_profile_read(pg2_engine* e, float ms_out[3], int64_t* steps) {
    EngineBase* b = e->impl.get();
    DeviceGuard guard__(b->device);
    b->prof_collect();
    for (int k = 0; k < 3; k++) ms_out[k] = (float)b->prof_ms[k];
    if (steps) *steps = b->prof_steps;
    return 0;
}

int64_t pg2_read_field(pg2_engine* e, const char* name, void* out, int64_t capacity, int32_t* elem_size, int32_t* per_env) {
    EngineBase* b = e->impl.get();
    void* ptr; int esz, pe;
    if (!b->find_field(name, &ptr, &esz, &pe)) { g_error = std::string("unknown field ") + name; return -1; }
    if (elem_size) *elem_size = esz;
    if (per_env) *per_env = pe;
    int64_t bytes = (int64_t)esz * pe * b->N;
    if (!out) return bytes;
    if (capacity < bytes) { g_error = "pg2_read_field: buffer too small"; return -2; }
    DeviceGuard guard__(b->device);
    cudaStreamSynchronize(b->stream);
    if (cudaMemcpy(out, ptr, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) { g_error = "pg2_read_field: copy failed"; return -3; }
    return bytes;
}

int64_t pg2_write_field(pg2_engine* e, const char* name, const void* in, int64_t bytes_in) {
    EngineBase* b = e->impl.get();
    void* ptr; int esz, pe;
    if (!b->find_field(name, &ptr, &esz, &pe)) { g_error = std::string("unknown field ") + name; return -1; }
    int64_t bytes = (int64_t)esz * pe * b->N;
    if (bytes_in != bytes) { g_error = "pg2_write_field: size mismatch"; return -2; }
    DeviceGuard guard__(b->device);
    cudaStreamSynchronize(b->stream);
    if (cudaMemcpy(ptr, in, bytes, cudaMemcpyHostToDevice) != cudaSuccess) { g_error = "pg2_write_field: copy failed"; return -3; }
    cudaMemset(b->common.view_valid, 0, (size_t)b->N);   // a tile map or camera may have changed: drop the cached views
    if (b->init_shadow()) return -3;                      // ... and the levels generated ahead of time (RNG state may have changed)
    return bytes;
}

// blob = header { magic, game tag, N, parity, state bytes, common bytes } + the sections of blob_sections, in order
struct SnapshotHeader { uint32_t magic, game; int32_t n, parity; uint64_t state_bytes, common_bytes; };
static const uint32_t SNAPSHOT_MAGIC = 0x50473253u;   // "PG2S"
struct BlobSection { void* dev; size_t bytes; };
static const int BLOB_SECTIONS = 7;

// The device buffers a blob holds: state_mem, common_mem and the current results (final_obs only when the engine has it:
// a blob restores only into an engine with the same setting, which the size check enforces). Returns the size of the
// blob; *nsec = the number of sections.
static int64_t blob_sections(EngineBase* b, BlobSection sec[BLOB_SECTIONS], int* nsec) {
    const EngineBase::Outputs& o = b->out[b->cur];
    const size_t n = (size_t)b->N;
    const BlobSection all[BLOB_SECTIONS] = { { b->state_mem, b->state_alloc_bytes() }, { b->common_mem, CommonState::bytes(b->N) },
                                             { o.obs, n * OBS_BYTES }, { o.reward, n * sizeof(float) }, { o.terminated, n }, { o.truncated, n },
                                             { o.final_obs, n * OBS_BYTES } };
    *nsec = b->final_on ? 7 : 6;
    int64_t total = sizeof(SnapshotHeader);
    for (int k = 0; k < *nsec; k++) { sec[k] = all[k]; total += (int64_t)all[k].bytes; }
    return total;
}

int64_t pg2_snapshot(pg2_engine* e, void* out, int64_t capacity) {
    EngineBase* b = e->impl.get();
    BlobSection sec[BLOB_SECTIONS];
    int nsec = 0;
    const int64_t total = blob_sections(b, sec, &nsec);
    if (!out) return total;
    if (capacity < total) { g_error = "pg2_snapshot: buffer too small"; return -2; }
    if (b->pipelined) { g_error = "pg2_snapshot: flush the pipelined stepping first (pg2_pipeline_flush) and use pg2_step"; return -2; }
    DeviceGuard guard__(b->device);
    if (cudaStreamSynchronize(b->stream) != cudaSuccess) { g_error = "pg2_snapshot: sync failed"; return -3; }
    SnapshotHeader h{ SNAPSHOT_MAGIC, b->game_tag(), b->N, b->parity, (uint64_t)sec[0].bytes, (uint64_t)sec[1].bytes };
    char* p = (char*)out;
    memcpy(p, &h, sizeof(h)); p += sizeof(h);
    bool ok = true;
    for (int k = 0; k < nsec; k++) { ok = ok && cudaMemcpy(p, sec[k].dev, sec[k].bytes, cudaMemcpyDeviceToHost) == cudaSuccess; p += sec[k].bytes; }
    if (!ok) { g_error = "pg2_snapshot: copy failed"; return -3; }
    return total;
}

int64_t pg2_restore(pg2_engine* e, const void* blob, int64_t bytes) {
    EngineBase* b = e->impl.get();
    BlobSection sec[BLOB_SECTIONS];
    int nsec = 0;
    const int64_t total = blob_sections(b, sec, &nsec);
    SnapshotHeader h;
    if (bytes < (int64_t)sizeof(h)) { g_error = "pg2_restore: truncated blob"; return -2; }
    memcpy(&h, blob, sizeof(h));
    if (h.magic != SNAPSHOT_MAGIC || h.game != b->game_tag() || h.n != b->N || h.state_bytes != sec[0].bytes || h.common_bytes != sec[1].bytes || bytes != total) {
        g_error = "pg2_restore: blob does not belong to this game / shard size"; return -2;
    }
    DeviceGuard guard__(b->device);
    if (cudaStreamSynchronize(b->stream) != cudaSuccess) { g_error = "pg2_restore: sync failed"; return -3; }
    const char* p = (const char*)blob + sizeof(h);
    bool ok = true;
    for (int k = 0; k < nsec; k++) { ok = ok && cudaMemcpy(sec[k].dev, p, sec[k].bytes, cudaMemcpyHostToDevice) == cudaSuccess; p += sec[k].bytes; }
    // the reset-list counters are transient within a step: zero them like a fresh engine, keep the parity of the snapshot
    ok = ok && cudaMemset(b->reset_count, 0, 4 * sizeof(int)) == cudaSuccess;
    if (b->final_ticket) ok = ok && cudaMemset(b->final_ticket, 0, 2 * sizeof(int)) == cudaSuccess;
    ok = ok && cudaMemset(b->common.view_valid, 0, (size_t)b->N) == cudaSuccess;   // the view caches are not part of the blob
    b->parity = h.parity;
    if (!ok) { g_error = "pg2_restore: copy failed"; return -3; }
    if (b->init_shadow()) return -3;   // the levels generated ahead of time are not part of the blob: regenerate them
    return total;
}

// Host-only (no CUDA call): texture `name` as the engine uploads it into the device atlas — RGBA8 texels, RGB textures with
// A = 255 — decoded from the packed blob by the product's own loader (assets.cpp). The build-container test compares it
// with the reference's PNG (tests/test_assets_blob.py). Returns the texel count, <0 on error; out may be NULL to query.
int64_t pg2_load_texture_host(const char* assets_path, const char* name, int32_t* w, int32_t* h, int32_t* blend, uint32_t* out, int64_t capacity) {
    std::vector<TexInfo> infos;
    std::vector<uint32_t> texels;
    std::string err;
    const char* names[1] = { name };
    if (!name || !load_textures(assets_path, names, 1, &infos, &texels, &err)) { g_error = err.empty() ? "pg2_load_texture_host: null name" : err; return -1; }
    if (w) *w = infos[0].w;
    if (h) *h = infos[0].h;
    if (blend) *blend = (int32_t)infos[0].blend;
    const size_t n = (size_t)infos[0].w * infos[0].h;   // the texture follows the atlas' black texel (atlas[0])
    if (out) {
        if (capacity < (int64_t)n) { g_error = "pg2_load_texture_host: buffer too small"; return -2; }
        memcpy(out, texels.data() + infos[0].offset, n * sizeof(uint32_t));
    }
    return (int64_t)n;
}

}  // extern "C"
