// Bodies of the three per-step kernels, shared between the __global__ entry points in
// engine.cu and the single-threaded test harness tests/hostsim/ (see pg2_platform.cuh), and the
// render kernels themselves, which tests/raster/ also instantiates for synthetic scenes.
#pragma once
#include "pg2_render.cuh"
#include "pg2_state.cuh"
#include "pg2_warp.cuh"

namespace pg2 {

// rng.seed(seed) + process-lifetime defaults (cenv_make)
PG2_TU_LOCAL PG2_DEV_NOINLINE void seed_body(const CommonState& c, int env, uint32_t seed, bool init_persistent) {
    mt_seed(c.mt + (size_t)env * MT_N, seed);
    c.mti[env] = MT_N;
    if (init_persistent) {
        c.cam_x[env] = 0.0f; c.cam_y[env] = 0.0f;   // Renderer::camera_position{0} (renderer.h:18)
        c.sprites_valid[env] = 0; c.ep_steps[env] = 0; c.fault[env] = 0; c.view_valid[env] = 0;
    }
}

// cenv_step for one env (without the render): returns "episode over" (terminated or truncated)
template <class G>
PG2_DEV bool step_body(const typename G::State& s, const CommonState& c, int env, int action, float* reward,
                       uint8_t* terminated, uint8_t* truncated, int max_episode_steps, const StepCtx& ctx) {
    float r = 0.0f;
    bool term = false;
    if (G::LANE_AWARE || ctx.nlanes == 1) {
        term = G::step(s, c, env, action, &r, ctx);
    } else {   // the game's step is single-threaded: the warp's leader runs it, the result is broadcast
        if (ctx.leader()) term = G::step(s, c, env, action, &r, StepCtx{ 0, 1 });
        __syncwarp();
        term = warp_bcast((int)term) != 0;
        r = warp_bcast(r);
    }
    bool trunc = false;
    int ep = c.ep_steps[env] + 1;
    if (max_episode_steps > 0 && ep >= max_episode_steps && !term) trunc = true;
    ctx.sync();
    if (ctx.leader()) {
        c.ep_steps[env] = ep;
        reward[env] = r;
        terminated[env] = term ? 1 : 0;
        truncated[env] = trunc ? 1 : 0;
    }
    return term || trunc;
}

// reset() for one env by one warp; `mt` = 624 words of per-warp scratch, `arena` = G::RESET_ARENA bytes
template <class G>
PG2_DEV void reset_body(const typename G::State& s, const CommonState& c, int env, uint32_t* mt, char* arena, int lane) {
    uint32_t* gmt = c.mt + (size_t)env * MT_N;
    for (int i = lane; i < MT_N; i += WARP_LANES) mt[i] = gmt[i];
    __syncwarp();
    WarpCtx ctx;
    ctx.rng.mt = mt; ctx.rng.idx = c.mti[env]; ctx.rng.lane = lane;
    ctx.lane = lane; ctx.arena = arena; ctx.arena_off = 0; ctx.arena_cap = G::RESET_ARENA;
    ctx.mode = c.mode < 0 ? G::DEFAULT_MODE : c.mode;
    G::regenerate(s, c, env, ctx);
    __syncwarp();
    for (int i = lane; i < MT_N; i += WARP_LANES) gmt[i] = mt[i];
    if (lane == 0) { c.mti[env] = ctx.rng.idx; c.ep_steps[env] = 0; c.view_valid[env] = 0; }   // new level: the cached view is stale
    __syncwarp();
}

// Debug build (-DPG2_PHASE_TIMERS): wall cycles of the render phases of a frame, as seen by thread 0 of the CTA, summed over
// all frames: [0] frames, [1] ticket + frame_begin, [2] build_frame, [3] finalize, [4] rasterise (thread 0's warp).
#ifdef PG2_PHASE_TIMERS
__device__ unsigned long long g_phase[8];
#define PG2_PHASE_MARK(k) do { if (threadIdx.x == 0) { long long now__ = clock64(); atomicAdd(&g_phase[k], (unsigned long long)(now__ - phase_t__)); phase_t__ = now__; } } while (0)
#else
#define PG2_PHASE_MARK(k) do { } while (0)
#endif

template <class G>
using FrameOf = FrameT<G::MAX_POST, G::ROTATES, G::TILE_CLASSES, G::WIN_ROWS, G::BLIT_UNROLL>;

// render_game(true) + RGBA->RGB pack for one env by one CTA (f.tileword filled by frame_init_tiletex before).
// view_cache (G::STATIC_VIEW games, else nullptr): VIEW_CACHE_BYTES per env = the env's base image;
// c.view_valid[env] says whether it is current.
template <class G>
PG2_DEV void render_body(const typename G::State& s, const CommonState& c, int env, FrameOf<G>& f, const TexInfo* __restrict__ tex,
                         const uint32_t* __restrict__ atlas, uint8_t* __restrict__ obs, uint8_t* __restrict__ view_cache = nullptr,
                         bool begin_and_sync = true) {
    uint8_t* cache = (G::STATIC_VIEW && view_cache) ? view_cache + (size_t)env * VIEW_CACHE_BYTES : nullptr;
    if (begin_and_sync) {
        frame_begin(f, cache != nullptr && c.view_valid[env] != 0);
        __syncthreads();
    }
#ifdef PG2_PHASE_TIMERS
    long long phase_t__ = clock64();
#endif
    G::build_frame(s, c, env, f, tex);
    __syncthreads();   // the only barrier between the frame builder's smem writes and their readers
    PG2_PHASE_MARK(2);
    frame_finalize<G>(f);
    PG2_PHASE_MARK(3);
    // a frame that needs the general ordered path everywhere (never observed) is neither cached nor marked
    uint8_t* img = (cache && (f.reuse || !f.wide)) ? cache : nullptr;
    frame_rasterise<G>(f, atlas, obs + (size_t)env * OBS_BYTES, img);
    PG2_PHASE_MARK(4);
    if (img && !f.reuse && threadIdx.x == 0) c.view_valid[env] = 1;   // read by later launches only
    if (f.overflow && threadIdx.x == 0) c.fault[env] |= 8;            // tile window taller than G::WIN_ROWS: the frame is wrong
}

// render_game(false) + the RGB read-out of cenv_render (coinrun.cpp:393-411, 443-470) for ONE env: a frame of any size
// with the window size as camera_size, drawn pixel by pixel along the general ordered path (cold path: the human
// viewer). Every CTA of the launch describes the frame for itself and shades the pixels [first, last) of the
// row-major frame; out = width * height * 3 bytes. Returns false when the window spans more tile rows than the frame
// tables hold (G::WIN_ROWS): rows beyond them are missing from the frame, and the caller must report it as an error.
template <class G>
PG2_DEV bool render_human_body(const typename G::State& s, const CommonState& c, int env, FrameOf<G>& f, const TexInfo* __restrict__ tex,
                               const uint32_t* __restrict__ atlas, uint8_t* __restrict__ out, int width, int height, int first, int last) {
    frame_begin(f, false);
    __syncthreads();
    if (threadIdx.x == 0) { f.view_w = (float)width; f.view_h = (float)height; f.human = 1; }
    __syncthreads();
    G::build_frame(s, c, env, f, tex);
    __syncthreads();
    frame_finalize<G>(f);
    for (int p = first + (int)threadIdx.x; p < last; p += CTA_THREADS) {
        const uint32_t color = shade_human_pixel<G>(f, atlas, p % width, p / width);
        out[3 * (size_t)p] = (uint8_t)color; out[3 * (size_t)p + 1] = (uint8_t)(color >> 8); out[3 * (size_t)p + 2] = (uint8_t)(color >> 16);
    }
    return f.overflow == 0;
}

#ifndef PG2_HOSTSIM
// ---- __global__ entry points of the render (instantiated by engine.cu, and by tests/raster/ for synthetic scenes)

// Level prefetch (G::PREFETCH_LEVELS): the NEXT level of every env is generated one episode ahead into a shadow copy of the
// state (k_reset on the shadow state, asynchronous, second stream). When an env finishes, k_step makes sure that level exists
// (swap_wait) and flags the env in `pending`; the render CTA that draws the env copies the shadow's reset-written fields over
// the live ones first (swap_copy), and the env goes onto the generator's list, which prepares the level after that. Field
// table: one entry per copied SoA field.
struct SwapField { char* live; const char* shadow; int esz, per_env, env_major; };
constexpr int MAX_SWAP_FIELDS = 64;
struct SwapTable { SwapField f[MAX_SWAP_FIELDS]; int n; };
struct SwapArgs {
    SwapTable table;          // table.n == 0: no level prefetch
    CommonState shadow_c;
    const int* gen_done;      // [N] levels delivered by the generator (beyond the first)
    int* used;                // [N] levels taken
};

// k_render, the whole CTA that is about to draw a finished env: copy the reset-written fields shadow -> live. Loads are issued
// in batches before their stores (the compiler cannot prove that a store does not alias the next load, which would
// serialise one memory round trip per element): short fields (<= blockDim elements per env) eight fields per round, one
// element per thread; long ones (tile map, MT19937 words, particle pools) eight elements per thread per round.
PG2_TU_LOCAL __device__ __noinline__ void swap_copy(const SwapArgs& a, const CommonState& live_c, int env, int N) {
    const int tid = threadIdx.x, nthr = CTA_THREADS;   // called by the render CTA
    __threadfence();
    auto elem_off = [&](const SwapField& f, int j) { return f.env_major ? ((size_t)env * f.per_env + j) * f.esz : ((size_t)j * N + env) * f.esz; };
    for (int i0 = 0; i0 < a.table.n; i0 += 8) {
        uint32_t v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            v[k] = 0u;
            if (i0 + k >= a.table.n) continue;
            const SwapField f = a.table.f[i0 + k];
            if (f.per_env > nthr || tid >= f.per_env || (f.esz != 4 && f.esz != 1)) continue;
            const size_t off = elem_off(f, tid);
            v[k] = f.esz == 4 ? *(const uint32_t*)(f.shadow + off) : (uint32_t)(uint8_t)f.shadow[off];
        }
#pragma unroll
        for (int k = 0; k < 8; k++) {
            if (i0 + k >= a.table.n) continue;
            const SwapField f = a.table.f[i0 + k];
            if (f.per_env > nthr || tid >= f.per_env || (f.esz != 4 && f.esz != 1)) continue;
            const size_t off = elem_off(f, tid);
            if (f.esz == 4) *(uint32_t*)(f.live + off) = v[k]; else f.live[off] = (char)v[k];
        }
    }
    for (int i = 0; i < a.table.n; i++) {
        const SwapField f = a.table.f[i];
        if (f.per_env <= nthr && (f.esz == 4 || f.esz == 1)) continue;
        if (f.esz != 4 && f.esz != 1) {   // other element sizes, byte by byte (jumper's uint16_t spike_cell)
            for (int j = tid; j < f.per_env; j += nthr) { const size_t off = elem_off(f, j); for (int bb = 0; bb < f.esz; bb++) f.live[off + bb] = f.shadow[off + bb]; }
            continue;
        }
        // an env-major byte field whose per-env block is word-aligned is copied as words
        const bool as_words = f.env_major && f.esz == 1 && ((((size_t)env * f.per_env) | (size_t)f.per_env | (size_t)(uintptr_t)f.live | (size_t)(uintptr_t)f.shadow) & 3) == 0;
        const int count = as_words ? f.per_env / 4 : f.per_env, esz = as_words ? 4 : f.esz;
        for (int j0 = 0; j0 < count; j0 += 8 * nthr) {
            uint32_t u[8];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const int j = j0 + q * nthr + tid;
                const size_t off = f.env_major ? ((size_t)env * f.per_env * f.esz + (size_t)j * esz) : ((size_t)j * N + env) * esz;
                u[q] = j >= count ? 0u : esz == 4 ? *(const uint32_t*)(f.shadow + off) : (uint32_t)(uint8_t)f.shadow[off];
            }
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const int j = j0 + q * nthr + tid;
                const size_t off = f.env_major ? ((size_t)env * f.per_env * f.esz + (size_t)j * esz) : ((size_t)j * N + env) * esz;
                if (j < count) { if (esz == 4) *(uint32_t*)(f.live + off) = u[q]; else f.live[off] = (char)u[q]; }
            }
        }
    }
    if (tid == 0) {   // what reset_body does besides the level
        a.used[env] += 1;   // read by this env's next wait only
        live_c.ep_steps[env] = 0; live_c.view_valid[env] = 0;
        live_c.fault[env] |= a.shadow_c.fault[env];
    }
    __syncthreads();   // the CTA reads what it just wrote
}

// Persistent CTAs; frames are handed out through a ticket counter, so a CTA that drew cheap frames simply takes
// more of them. mode 0: every env; mode 1: every env that is NOT being reset this step (k_reset runs concurrently
// on a second stream); mode 2: exactly the envs of the reset list (after k_reset).
// FINAL: the render of an engine created with final_obs (Engine::final_on), which returns the terminal frame of every env
// that finishes. Two uses:
//   - level prefetch, mode 0 with the swap list: the CTA of a finished env draws two frames, first the terminal frame from
//     the state the episode ended in into final_obs (a static-view game may load its cached base image: it is still the
//     episode's own), then, after the level swap, the reset frame into obs;
//   - inline reset, mode 2 over the reset list between k_step and k_reset: obs = the terminal frames, no swap.
// Block 0 zeroes *zero_ticket when given: the ticket of the next such launch. Without FINAL, final_obs and zero_ticket are
// ignored. The FINAL instances are compiled in their own translation unit (engine_final.cu): instantiated beside the others,
// they change the code of every k_render<G, false>, the kernels of every engine without final_obs.
template <class G, bool FINAL>
__global__ void __launch_bounds__(RENDER_THREADS, G::RENDER_MIN_CTAS) k_render(typename G::State s, CommonState c, const TexInfo* __restrict__ tex,
                                                           const uint32_t* __restrict__ atlas, uint8_t* __restrict__ obs,
                                                           int* __restrict__ ticket, int mode, const int* __restrict__ list,
                                                           const int* __restrict__ list_count, const uint8_t* __restrict__ pending, int N,
                                                           uint8_t* __restrict__ view_cache, const __grid_constant__ SwapArgs swap,
                                                           uint8_t* __restrict__ final_obs, int* __restrict__ zero_ticket) {
    __shared__ FrameOf<G> f;
    __shared__ int s_env;
    if constexpr (FINAL) { if (zero_ticket != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *zero_ticket = 0; }
    const int count = mode == 2 ? *list_count : N;
    frame_init_tiletex<G>(f, tex);
    // thread 0: the next frame's env (-1: none left) and whether its cached base image is valid — both fetched one frame
    // ahead, so that their memory round trips overlap the current frame's work (an env's view_valid only changes when the
    // env itself is rendered, or in earlier kernels)
    __shared__ int s_swap;
    int next_env = -1;
    bool next_reuse = false, next_swap = false;
    // level prefetch: the envs that finished in this step (the list k_step appended them to) come first — their CTAs copy the
    // next level in before drawing, which must not land in the kernel's tail — then every env that is not on the list
    const int nfirst = (swap.table.n > 0 && mode == 0) ? *list_count : 0;
    auto take_ticket = [&]() {
        int t = atomicAdd(ticket, 1);
        if (nfirst > 0) {
            if (t < nfirst) {   // FINAL: the first frame of a finished env is its terminal frame, drawn before the swap
                next_env = list[t]; next_swap = true;
                next_reuse = FINAL && G::STATIC_VIEW && view_cache != nullptr && c.view_valid[next_env] != 0;
                return;
            }
            t -= nfirst;
            while (t < count && pending[t]) t = atomicAdd(ticket, 1) - nfirst;
        }
        if (!FINAL && mode == 1) while (t < count && pending[t]) t = atomicAdd(ticket, 1);   // FINAL never runs mode 1: keep the loop out of its code
        next_env = t < count ? (mode == 2 ? list[t] : t) : -1;
        next_swap = false;
        next_reuse = G::STATIC_VIEW && view_cache != nullptr && next_env >= 0 && !next_swap && c.view_valid[next_env] != 0;
    };
    if (threadIdx.x == 0) take_ticket();
    for (;;) {
#ifdef PG2_PHASE_TIMERS
        long long phase_t__ = clock64();
#endif
        __syncthreads();   // every warp is done with the previous frame (bands are stored per warp, without a CTA barrier)
        if (threadIdx.x == 0) { s_env = next_env; s_swap = next_swap ? 1 : 0; }
        frame_begin(f, next_reuse);
        __syncthreads();
        const int env = s_env;
        if (env < 0) break;
        PG2_PHASE_MARK(1);
#ifdef PG2_PHASE_TIMERS
        if (threadIdx.x == 0) atomicAdd(&g_phase[0], 1ull);
#endif
        // the next frame's ticket is taken now: the atomic's round trip overlaps this frame's work
        const bool do_swap = s_swap != 0;
        if (threadIdx.x == 0) take_ticket();
        if constexpr (FINAL) {
            // one render_body call site for both frames of a finished env: a second inlined copy spills registers
            uint8_t* dst = do_swap ? final_obs : obs;
            for (;;) {
                render_body<G>(s, c, env, f, tex, atlas, dst, view_cache, false);
                if (dst == obs) break;
                __syncthreads();   // the same barriers as between two frames of the loop
                frame_begin(f, false);
                __syncthreads();
                swap_copy(swap, c, env, N);
                dst = obs;
            }
        } else {
            if (do_swap) swap_copy(swap, c, env, N);
            render_body<G>(s, c, env, f, tex, atlas, obs, view_cache, false);
        }
    }
    if ((threadIdx.x & 31) == 0) frame_store_wait();   // every warp issued bulk stores of its own
}

// Human-mode frame of one env (cenv_render): every CTA shades a contiguous slice of the width x height frame.
// *overflow (zeroed by the caller) is set when the frame is incomplete (render_human_body).
template <class G>
__global__ void __launch_bounds__(RENDER_THREADS) k_render_human(typename G::State s, CommonState c, int env, const TexInfo* __restrict__ tex,
                                                                 const uint32_t* __restrict__ atlas, uint8_t* __restrict__ out, int width, int height,
                                                                 int* __restrict__ overflow) {
    __shared__ FrameOf<G> f;
    frame_init_tiletex<G>(f, tex);
    const int total = width * height, per = (total + gridDim.x - 1) / gridDim.x;
    const int first = blockIdx.x * per, last = min(total, first + per);
    if (!render_human_body<G>(s, c, env, f, tex, atlas, out, width, height, first, last) && threadIdx.x == 0) *overflow = 1;
}
#endif  // PG2_HOSTSIM

}  // namespace pg2
