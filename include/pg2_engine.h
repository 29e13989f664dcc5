/* procgen2-b200 — C ABI of the batched, GPU-resident environment engine.
 *
 * Plain C: pointers and sizes only, no torch / CUDA types in the signatures. The per-game
 * drop-in libraries (libCoinRun.so, libMaze.so, ... — same file names as the reference's CMake
 * targets, games/<g>/CMakeLists.txt `add_library(<Game> SHARED ...)`) implement the reference's
 * cenv ABI (include/cenv.h) on top of these entry points; Python front-ends bind them with
 * ctypes (procgen2_b200/engine.py).
 *
 * What each call replaces in the reference (one environment per process there, N here):
 *   pg2_create  <- cenv_make   games/coinrun/coinrun.cpp:127-306 (maze.cpp:85, bossfight.cpp:…)
 *   pg2_reset   <- cenv_reset  games/coinrun/coinrun.cpp:308-339
 *   pg2_step*   <- cenv_step   games/coinrun/coinrun.cpp:341-391 (+ caller-side
 *                  "if terminated: reset" of game_test.py:38-40, done on device as auto-reset)
 *   pg2_fetch   <- the observation / reward / terminated read-out of cenv/cenv.py:289-309
 *   pg2_destroy <- cenv_close  games/coinrun/coinrun.cpp:413-441
 *
 * Environment i of an engine created with (seed, first_env) is seeded `seed + first_env + i`
 * and reproduces, bit for bit, a reference process created with that seed
 * (cenv_make(seed) -> cenv_reset() -> cenv_step()* with reset-on-terminate).
 *
 * All functions return 0 on success, non-zero on error (pg2_last_error() gives the text) —
 * the same convention as the cenv entry points (cenv/cenv.py:208-209).
 */
#ifndef PG2_ENGINE_H
#define PG2_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PG2_API __attribute__((__visibility__("default")))

typedef struct pg2_engine pg2_engine;

typedef struct {
    const char* game;            /* "maze" | "coinrun" | "bossfight" | "chaser" | "climber" | "caveflyer" | "jumper" */
    int32_t num_envs;            /* environments owned by this engine (this GPU's shard) */
    int32_t seed;                /* base seed; env i gets seed + first_env + i (uint32 wrap) */
    int32_t first_env;           /* global index of this shard's first environment */
    int32_t device;              /* CUDA device ordinal */
    int32_t max_episode_steps;   /* extension: >0 truncates episodes (SURVEY Q23); 0 = reference behaviour */
    const char* assets_path;     /* packed asset blob; NULL -> $PG2_ASSETS or <lib dir>/../data/assets.bin */
    int32_t auto_reset;          /* 1: finished envs run reset() on device inside the same step (observation =
                                    reset frame); 0: reference behaviour, the caller calls pg2_reset */
    int32_t distribution_mode;   /* level-generator mode of the game's tilemap Config (games/<g>/tilemap.h: compile-time in
                                    the reference): -1 = the reference's default, 0 easy, 1 hard, 2 memory / extreme.
                                    Every mode of a game's enum is built (maze / chaser / jumper / caveflyer 0-2, coinrun /
                                    climber / bossfight 0-1); a mode the game does not have makes pg2_create fail */
    int32_t final_obs;           /* 1: also return the terminal frame of every env that finishes (Gymnasium's final_obs):
                                    row e of pg2_final_obs_device is written in a step iff env e terminated or was truncated
                                    in it, with render_game(true) of the state it finished in — what an auto_reset = 0 engine
                                    returns as that step's observation. Other rows keep older contents (zero at creation);
                                    pg2_reset does not write any. obs, reward, flags and state are the same as with 0.
                                    Needs auto_reset = 1 (pg2_create fails otherwise). 0 = off: no buffer, no extra work */
} pg2_config;

PG2_API int32_t pg2_create(const pg2_config* cfg, pg2_engine** out);
PG2_API void pg2_destroy(pg2_engine* e);

/* cenv_reset for every environment. seeds: NULL (continue the RNG streams) or num_envs host
 * int32 (option "seed" of cenv_reset: reseed env i with seeds[i]). Renders the reset frame. */
PG2_API int32_t pg2_reset(pg2_engine* e, const int32_t* seeds);

/* One cenv_step for every environment. `actions` = num_envs int32 in HOST memory (copied to
 * the device inside the call) / DEVICE memory. Asynchronous: results stay in HBM. */
PG2_API int32_t pg2_step(pg2_engine* e, const int32_t* actions_host);
PG2_API int32_t pg2_step_device(pg2_engine* e, const int32_t* actions_device);

/* cenv_render (games/coinrun/coinrun.cpp:393-411): environment `env`'s current scene drawn again at width x height with the
 * window size as camera_size (render_game(false): camera_scale = game_zoom * width / 64), as width * height * 3 RGB
 * bytes (row-major) in HOST memory. A cold path for the human viewer; synchronous.
 * Fails (nonzero, pg2_last_error) rather than return an incomplete frame when width or height exceeds 32767 pixels (blit
 * rects are 16-bit pixel coordinates) or when the window spans more tile rows than the game's frame tables hold
 * (WIN_ROWS: a window much taller than wide; e.g. maze at 64 x 4096). */
PG2_API int32_t pg2_render_human(pg2_engine* e, int32_t env, int32_t width, int32_t height, uint8_t* out_rgb);

/* Copy results of the last step/reset to host buffers (any pointer may be NULL) and wait.
 * obs: num_envs*12288 uint8 (64x64x3 RGB, row-major), reward: num_envs float,
 * terminated / truncated: num_envs uint8. */
PG2_API int32_t pg2_fetch(pg2_engine* e, uint8_t* obs, float* reward, uint8_t* terminated, uint8_t* truncated);

/* pg2_fetch without the wait: copies enqueued on the engine's stream, completed by pg2_sync (asynchronous only into
 * page-locked memory). pg2_host_alloc / pg2_host_free: page-locked host memory for such buffers (NULL on failure). */
PG2_API int32_t pg2_fetch_async(pg2_engine* e, uint8_t* obs, float* reward, uint8_t* terminated, uint8_t* truncated);
PG2_API void* pg2_host_alloc(size_t bytes);
PG2_API void pg2_host_free(void* p);

/* Depth-1 pipelined stepping for host-buffer callers: enqueues step t (H2D of its actions, the kernels, D2H of
 * its results into the given host buffers — pinned for true overlap — on a second stream) and returns when the
 * results of step t-1, written to the buffers passed to the PREVIOUS call, are complete. Alternate two sets of
 * host buffers; pg2_pipeline_flush() completes the last step. The HBM outputs are double-buffered from the first
 * call on, so pg2_*_device() pointers alternate between two buffers in this mode. */
PG2_API int32_t pg2_step_pipelined(pg2_engine* e, const int32_t* actions_host, uint8_t* obs, float* reward,
                                   uint8_t* terminated, uint8_t* truncated);
PG2_API int32_t pg2_pipeline_flush(pg2_engine* e);

/* Device-resident results (valid until the next step on the engine's stream). */
PG2_API uint8_t* pg2_obs_device(pg2_engine* e);
PG2_API float* pg2_reward_device(pg2_engine* e);
PG2_API uint8_t* pg2_terminated_device(pg2_engine* e);
PG2_API uint8_t* pg2_truncated_device(pg2_engine* e);
/* final_obs engines: the terminal frames, num_envs * 12288 uint8 like obs (NULL when final_obs is off). */
PG2_API uint8_t* pg2_final_obs_device(pg2_engine* e);

/* final_obs engines: copy the terminal-frame buffer to host memory and wait (pg2_fetch_final), or enqueue the copies of
 * the rows with rows[i] != 0 (rows: num_envs host flags, NULL = every row) to the same offsets of `host`, one copy per run
 * of consecutive rows, completed by pg2_sync (pg2_fetch_final_async). Fail on an engine without final_obs. */
PG2_API int32_t pg2_fetch_final(pg2_engine* e, uint8_t* host);
PG2_API int32_t pg2_fetch_final_async(pg2_engine* e, const uint8_t* rows, uint8_t* host);

PG2_API int32_t pg2_sync(pg2_engine* e);
PG2_API void* pg2_stream(pg2_engine* e);            /* cudaStream_t the engine launches on */
PG2_API int32_t pg2_num_envs(pg2_engine* e);
PG2_API int32_t pg2_debug_phases(pg2_engine* e, uint64_t out[8]);   /* -DPG2_PHASE_TIMERS builds: render phase cycle counters; else -1 */
PG2_API int32_t pg2_step_epw(pg2_engine* e);        /* environments per warp in the step kernel (1 = a whole warp per env) */
PG2_API int64_t pg2_kernel_launches(pg2_engine* e); /* kernels launched so far (bench.py gpu_launches) */
PG2_API int64_t pg2_state_bytes_per_env(pg2_engine* e);

/* Per-kernel device timing (CUDA events on the engine's stream around each launch of
 * pg2_step*). enable != 0 starts/clears accumulation; pg2_profile_read synchronises and returns
 * accumulated milliseconds {step logic, level generation, render} and the number of steps. */
PG2_API int32_t pg2_profile(pg2_engine* e, int32_t enable);
PG2_API int32_t pg2_profile_read(pg2_engine* e, float ms_out[3], int64_t* steps);

/* Test / checkpoint access to the structure-of-arrays state: copies field `name` of the game
 * (or common) state to host memory. Returns bytes written, or <0 if the field is unknown or
 * `capacity` is too small. per_env receives the element count per environment. */
PG2_API int64_t pg2_read_field(pg2_engine* e, const char* name, void* out, int64_t capacity, int32_t* elem_size, int32_t* per_env);
PG2_API int64_t pg2_write_field(pg2_engine* e, const char* name, const void* in, int64_t bytes);

/* Snapshot / restore of the complete simulation state of the shard (every SoA field incl. the MT19937 streams, the
 * current observations / rewards / done flags, and the terminal frames of a final_obs engine): a checkpoint the reference
 * cannot take (SURVEY.md §5, §8f rank 4). pg2_snapshot(e, NULL, 0) returns the blob size; otherwise bytes written, <0 on
 * error. A blob restores only into an engine of the same game, shard size and final_obs setting. Stepping after pg2_restore reproduces the steps after pg2_snapshot bit for bit. */
PG2_API int64_t pg2_snapshot(pg2_engine* e, void* out, int64_t capacity);
PG2_API int64_t pg2_restore(pg2_engine* e, const void* blob, int64_t bytes);

/* Host-only helper (no CUDA call, works without a GPU): texture `name` (an "assets/..." path of the reference) exactly as
 * the engine uploads it into its device atlas — w*h RGBA8 texels (little-endian R,G,B,A; opaque RGB textures carry A = 255),
 * blend = 1 for alpha textures. Replaces Asset_Texture::load (games/coinrun/common_assets.cpp:3-17) for inspection:
 * the build-container test compares it with the PNG decoded by PIL. Returns the texel count (out may be NULL), <0 on error. */
PG2_API int64_t pg2_load_texture_host(const char* assets_path, const char* name, int32_t* w, int32_t* h, int32_t* blend,
                                      uint32_t* out, int64_t capacity);

PG2_API const char* pg2_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
