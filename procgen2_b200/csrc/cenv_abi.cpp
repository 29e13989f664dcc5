// cenv drop-in: one shared library per game (libMaze.so, libCoinRun.so, ...) exporting exactly
// the symbols of include/cenv.h, implemented on the batched GPU engine (include/pg2_engine.h).
// Compiled once per game with -DPG2_GAME="<game>".
//
// Mirrors the reference glue games/<g>/<g>.cpp:
//   cenv_make   option parsing "seed" | "width" | "height", space/obs buffers (coinrun.cpp:127-203)
//   cenv_reset  optional "seed" option, reset(), render, copy observation   (coinrun.cpp:308-339)
//   cenv_step   key "action" INT, step, render, copy observation            (coinrun.cpp:341-391)
//   cenv_close  frees the library-owned buffers                             (coinrun.cpp:413-441)
// Extension (documented in include/cenv.h): "num_envs", "device", "num_devices", "max_episode_steps", "auto_reset",
// "host_copy", "final_observation" make-options; batched "action"/"screen" buffers; per-env results and the DEVICE addresses of the
// result buffers as step / reset infos (+ the exported getter cenv_device_buffer). Host result buffers are pinned.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <string>
#include <vector>

#include "cenv.h"
#include "pg2_engine.h"

#ifndef PG2_GAME
#error "compile with -DPG2_GAME=\"<game>\""
#endif

static_assert(sizeof(cenv_key_value) == 24 && offsetof(cenv_key_value, value_buffer) == 16, "cenv_key_value layout");
static_assert(sizeof(cenv_option) == 24 && offsetof(cenv_option, value) == 16, "cenv_option layout");
static_assert(sizeof(cenv_step_data) == 40 && offsetof(cenv_step_data, terminated) == 24 && offsetof(cenv_step_data, truncated) == 25 &&
              offsetof(cenv_step_data, infos_size) == 28 && offsetof(cenv_step_data, infos) == 32, "cenv_step_data layout");

extern "C" {
CENV_API cenv_make_data make_data;
CENV_API cenv_reset_data reset_data;
CENV_API cenv_step_data step_data;
CENV_API cenv_render_data render_data;
}

namespace {

const int kVersion = 100;        // coinrun.cpp:9
const int kObsBytes = 64 * 64 * 3;
const int kNumActions = 15;      // coinrun.cpp:27

// One engine per device: shard d owns the contiguous env slice [g_first[d], g_first[d] + g_count[d]) (SURVEY §8e);
// seeds stay seed + global env index, so results do not depend on the number of devices.
std::vector<pg2_engine*> g_engines;
std::vector<int> g_first, g_count;
pg2_engine* g_engine = nullptr;   // == g_engines[0] (non-null <=> made)
int g_num_envs = 1;
int g_window_w = 512, g_window_h = 512;   // cenv_render's window (options "width" / "height"; limits: pg2_render_human)

int g_host_copy = 1;              // make-option "host_copy": 0 = observations stay in HBM (read them through the device pointers)
int g_final = 0;                  // make-option "final_observation": the terminal frames of finished envs as step infos

cenv_key_value g_observation;    // shared by reset_data and step_data, like the reference
cenv_key_value g_obs_space, g_act_space;
enum { INFO_REWARD, INFO_TERMINATED, INFO_TRUNCATED, INFO_SCREEN_DEV, INFO_REWARD_DEV, INFO_TERMINATED_DEV, INFO_TRUNCATED_DEV, INFO_STREAM, NUM_INFOS,
       INFO_FINAL_SCREEN_DEV = NUM_INFOS, INFO_FINAL_SCREEN };   // the last two: step infos with "final_observation" only
cenv_key_value g_infos[NUM_INFOS + 2];
float g_box[2] = { 0.0f, 255.0f };
int32_t g_nvec[1] = { kNumActions };
// host result buffers: page-locked (pg2_host_alloc), so the device -> host copies run at full PCIe speed and asynchronously
uint8_t *g_obs = nullptr, *g_term = nullptr, *g_trunc = nullptr, *g_final_obs = nullptr;
float* g_reward = nullptr;
std::vector<uint8_t> g_done;        // "final_observation": terminated | truncated of the last step, per env
std::vector<uint8_t> g_frame;
std::vector<int32_t> g_actions, g_seeds;
std::vector<int32_t> g_devptr[6];   // per info: (lo, hi) 32-bit halves of one address per device (the 6th: final_screen_device)

void free_host() {
    pg2_host_free(g_obs); pg2_host_free(g_reward); pg2_host_free(g_term); pg2_host_free(g_trunc); pg2_host_free(g_final_obs);
    g_obs = g_term = g_trunc = g_final_obs = nullptr; g_reward = nullptr;
}

// addresses of the device-resident results (they alternate between two buffer sets only in pg2_step_pipelined mode,
// which this library does not use: constant for the lifetime of the environment)
void publish_device_pointers() {
    for (int k = 0; k < 6; k++) g_devptr[k].assign(2 * g_engines.size(), 0);
    for (size_t d = 0; d < g_engines.size(); d++) {
        const void* p[6] = { pg2_obs_device(g_engines[d]), pg2_reward_device(g_engines[d]), pg2_terminated_device(g_engines[d]),
                             pg2_truncated_device(g_engines[d]), pg2_stream(g_engines[d]), pg2_final_obs_device(g_engines[d]) };
        for (int k = 0; k < 6; k++) {
            const uint64_t a = (uint64_t)(uintptr_t)p[k];
            g_devptr[k][2 * d] = (int32_t)(uint32_t)(a & 0xffffffffu);
            g_devptr[k][2 * d + 1] = (int32_t)(uint32_t)(a >> 32);
        }
    }
}

// results of the last step / reset -> host buffers. Every device's copies are enqueued first (asynchronous, pinned
// destination), then waited for: the transfers of different devices overlap.
int fetch() {
    for (size_t d = 0; d < g_engines.size(); d++) {
        const size_t o = (size_t)g_first[d];
        if (pg2_fetch_async(g_engines[d], g_host_copy ? g_obs + o * kObsBytes : nullptr, g_reward + o, g_term + o, g_trunc + o)) {
            fprintf(stderr, "[procgen2_b200] %s\n", pg2_last_error());
            return 1;
        }
    }
    for (size_t d = 0; d < g_engines.size(); d++)
        if (pg2_sync(g_engines[d])) { fprintf(stderr, "[procgen2_b200] %s\n", pg2_last_error()); return 1; }
    return 0;
}

// "final_observation" with host_copy, after fetch(): the terminal frames of the envs that finished in the step -> the host
// buffer, one copy per run of consecutive finished envs (the flags are on the host already); the other rows keep their
// older contents, as on the device.
int fetch_final() {
    for (int e = 0; e < g_num_envs; e++) g_done[e] = g_term[e] | g_trunc[e];
    for (size_t d = 0; d < g_engines.size(); d++) {
        const size_t o = (size_t)g_first[d];
        if (pg2_fetch_final_async(g_engines[d], g_done.data() + o, g_final_obs + o * kObsBytes)) {
            fprintf(stderr, "[procgen2_b200] %s\n", pg2_last_error());
            return 1;
        }
    }
    for (size_t d = 0; d < g_engines.size(); d++)
        if (pg2_sync(g_engines[d])) { fprintf(stderr, "[procgen2_b200] %s\n", pg2_last_error()); return 1; }
    return 0;
}

void destroy_all() {
    for (pg2_engine* e : g_engines) pg2_destroy(e);
    g_engines.clear(); g_first.clear(); g_count.clear();
    g_engine = nullptr;
    free_host();
}

}  // namespace

extern "C" {

int32_t cenv_get_env_version() { return kVersion; }

int32_t cenv_make(const char* /*render_mode*/, cenv_option* options, int32_t options_size) {
    destroy_all();
    unsigned int seed = (unsigned int)time(nullptr);     // coinrun.cpp:130
    int device = 0, num_devices = 1, max_episode_steps = 0, auto_reset = -1, distribution_mode = -1;
    g_num_envs = 1; g_host_copy = 1; g_final = 0;
    for (int i = 0; i < options_size; i++) {
        std::string name(options[i].name);
        if (options[i].value_type != CENV_VALUE_TYPE_INT) continue;
        int v = options[i].value.i;
        if (name == "seed") seed = (unsigned int)v;
        else if (name == "width") g_window_w = v;
        else if (name == "height") g_window_h = v;
        else if (name == "num_envs") g_num_envs = v;
        else if (name == "device") device = v;
        else if (name == "num_devices") num_devices = v;
        else if (name == "max_episode_steps") max_episode_steps = v;
        else if (name == "auto_reset") auto_reset = v;
        else if (name == "host_copy") g_host_copy = v != 0;
        else if (name == "distribution_mode") distribution_mode = v;
        else if (name == "final_observation") g_final = v != 0;
    }
    if (g_num_envs < 1 || (long long)g_num_envs * kObsBytes > 2147483647LL) {
        fprintf(stderr, "[procgen2_b200] num_envs out of range for an int32 cenv buffer size\n");
        return 1;
    }
    if (auto_reset < 0) auto_reset = g_num_envs > 1 ? 1 : 0;
    if (num_devices < 1 || num_devices > g_num_envs) {
        fprintf(stderr, "[procgen2_b200] num_devices must be in [1, num_envs]\n");
        return 1;
    }
    for (int d = 0, first = 0; d < num_devices; d++) {
        const int count = g_num_envs / num_devices + (d < g_num_envs % num_devices ? 1 : 0);
        pg2_config cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.game = PG2_GAME;
        cfg.num_envs = count;
        cfg.seed = (int32_t)seed;
        cfg.first_env = first;
        cfg.device = device + d;
        cfg.max_episode_steps = max_episode_steps;
        cfg.assets_path = nullptr;
        cfg.auto_reset = auto_reset;
        cfg.distribution_mode = distribution_mode;
        cfg.final_obs = g_final;
        pg2_engine* e = nullptr;
        if (pg2_create(&cfg, &e)) {
            fprintf(stderr, "[procgen2_b200] cenv_make failed (device %d): %s\n", device + d, pg2_last_error());
            destroy_all();
            return 1;
        }
        g_engines.push_back(e); g_first.push_back(first); g_count.push_back(count);
        first += count;
    }
    g_engine = g_engines[0];

    g_obs = (uint8_t*)pg2_host_alloc((size_t)g_num_envs * kObsBytes);
    g_reward = (float*)pg2_host_alloc(sizeof(float) * (size_t)g_num_envs);
    g_term = (uint8_t*)pg2_host_alloc((size_t)g_num_envs);
    g_trunc = (uint8_t*)pg2_host_alloc((size_t)g_num_envs);
    if (g_final && g_host_copy) {
        g_final_obs = (uint8_t*)pg2_host_alloc((size_t)g_num_envs * kObsBytes);
        if (g_final_obs) memset(g_final_obs, 0, (size_t)g_num_envs * kObsBytes);
    }
    g_done.assign(g_num_envs, 0);
    if (!g_obs || !g_reward || !g_term || !g_trunc || (g_final && g_host_copy && !g_final_obs)) {
        fprintf(stderr, "[procgen2_b200] cenv_make: cannot allocate the pinned host buffers: %s\n", pg2_last_error());
        destroy_all();
        return 1;
    }
    memset(g_obs, 0, (size_t)g_num_envs * kObsBytes); memset(g_reward, 0, sizeof(float) * (size_t)g_num_envs);
    memset(g_term, 0, (size_t)g_num_envs); memset(g_trunc, 0, (size_t)g_num_envs);
    publish_device_pointers();
    g_actions.assign(g_num_envs, 0);
    g_seeds.assign(g_num_envs, 0);
    g_frame.assign((size_t)g_window_w * g_window_h * 3, 0);

    g_obs_space = { "screen", CENV_SPACE_TYPE_BOX, 2, {} };
    g_obs_space.value_buffer.f = g_box;
    g_act_space = { "action", CENV_SPACE_TYPE_MULTI_DISCRETE, 1, {} };
    g_act_space.value_buffer.i = g_nvec;
    make_data.observation_spaces_size = 1;
    make_data.observation_spaces = &g_obs_space;
    make_data.action_spaces_size = 1;
    make_data.action_spaces = &g_act_space;

    g_observation = { "screen", CENV_VALUE_TYPE_BYTE, g_num_envs * kObsBytes, {} };
    g_observation.value_buffer.b = g_obs;

    reset_data.observations_size = 1;
    reset_data.observations = &g_observation;

    step_data.observations_size = 1;
    step_data.observations = &g_observation;
    step_data.reward.f = 0.0f;
    step_data.terminated = false;
    step_data.truncated = false;
    g_infos[INFO_REWARD] = { "reward", CENV_VALUE_TYPE_FLOAT, g_num_envs, {} };
    g_infos[INFO_REWARD].value_buffer.f = g_reward;
    g_infos[INFO_TERMINATED] = { "terminated", CENV_VALUE_TYPE_BYTE, g_num_envs, {} };
    g_infos[INFO_TERMINATED].value_buffer.b = g_term;
    g_infos[INFO_TRUNCATED] = { "truncated", CENV_VALUE_TYPE_BYTE, g_num_envs, {} };
    g_infos[INFO_TRUNCATED].value_buffer.b = g_trunc;
    static const char* const dev_keys[5] = { "screen_device", "reward_device", "terminated_device", "truncated_device", "stream" };
    for (int k = 0; k < 5; k++) {
        g_infos[INFO_SCREEN_DEV + k] = { dev_keys[k], CENV_VALUE_TYPE_INT, (int32_t)g_devptr[k].size(), {} };
        g_infos[INFO_SCREEN_DEV + k].value_buffer.i = g_devptr[k].data();
    }
    g_infos[INFO_FINAL_SCREEN_DEV] = { "final_screen_device", CENV_VALUE_TYPE_INT, (int32_t)g_devptr[5].size(), {} };
    g_infos[INFO_FINAL_SCREEN_DEV].value_buffer.i = g_devptr[5].data();
    g_infos[INFO_FINAL_SCREEN] = { "final_screen", CENV_VALUE_TYPE_BYTE, g_num_envs * kObsBytes, {} };
    g_infos[INFO_FINAL_SCREEN].value_buffer.b = g_final_obs;
    // the reference's single environment reports no infos (coinrun.cpp:200-202); the batched / device-resident
    // extension adds the per-env results and the device addresses (+ the terminal frames with "final_observation")
    const bool extended = g_num_envs > 1 || !g_host_copy || g_final;
    step_data.infos_size = extended ? NUM_INFOS + (g_final ? (g_host_copy ? 2 : 1) : 0) : 0;
    step_data.infos = extended ? g_infos : nullptr;
    reset_data.infos_size = extended ? 5 : 0;
    reset_data.infos = extended ? g_infos + INFO_SCREEN_DEV : nullptr;

    render_data.value_type = CENV_VALUE_TYPE_BYTE;
    render_data.value_buffer_width = g_window_w;
    render_data.value_buffer_height = g_window_h;
    render_data.value_buffer_channels = 3;
    render_data.value_buffer.b = g_frame.data();
    return 0;
}

int32_t cenv_reset(cenv_option* options, int32_t options_size) {
    if (!g_engine) return 1;
    bool reseed = false;
    for (int i = 0; i < options_size; i++) {
        std::string name(options[i].name);
        if (name == "seed" && options[i].value_type == CENV_VALUE_TYPE_INT) {
            // env i restarts its stream from seed + i (i = 0: exactly rng.seed(seed), coinrun.cpp:313-317)
            for (int e = 0; e < g_num_envs; e++) g_seeds[e] = (int32_t)((unsigned int)options[i].value.i + (unsigned int)e);
            reseed = true;
        }
    }
    for (size_t d = 0; d < g_engines.size(); d++)
        if (pg2_reset(g_engines[d], reseed ? g_seeds.data() + g_first[d] : nullptr)) {
            fprintf(stderr, "[procgen2_b200] cenv_reset failed: %s\n", pg2_last_error());
            return 1;
        }
    return fetch();
}

int32_t cenv_step(cenv_key_value* actions, int32_t actions_size) {
    if (!g_engine) return 1;
    std::fill(g_actions.begin(), g_actions.end(), 0);
    for (int i = 0; i < actions_size; i++) {
        std::string key(actions[i].key);
        if (key == "action") {
            if (actions[i].value_type != CENV_VALUE_TYPE_INT || actions[i].value_buffer_size != g_num_envs) {
                fprintf(stderr, "[procgen2_b200] cenv_step: \"action\" must be INT[%d]\n", g_num_envs);
                return 1;
            }
            memcpy(g_actions.data(), actions[i].value_buffer.i, sizeof(int32_t) * g_num_envs);
        }
    }
    // every device gets its slice of the actions and starts stepping (asynchronous launches); the fetches then
    // drain the devices one after the other while the others are still computing
    for (size_t d = 0; d < g_engines.size(); d++)
        if (pg2_step(g_engines[d], g_actions.data() + g_first[d])) {
            fprintf(stderr, "[procgen2_b200] cenv_step failed: %s\n", pg2_last_error());
            return 1;
        }
    if (fetch()) return 1;
    if (g_final && g_host_copy && fetch_final()) return 1;
    step_data.reward.f = g_reward[0];
    step_data.terminated = g_term[0] != 0;
    step_data.truncated = g_trunc[0] != 0;
    return 0;
}

// Human-mode frame: env 0's scene drawn again at window resolution with the window size as camera_size
// (render_game(false) + read-out, coinrun.cpp:393-411) — on the device (pg2_render_human).
int32_t cenv_render() {
    if (!g_engine) return 1;
    if (pg2_render_human(g_engine, 0, g_window_w, g_window_h, g_frame.data())) {
        fprintf(stderr, "[procgen2_b200] cenv_render failed: %s\n", pg2_last_error());
        return 1;
    }
    return 0;
}

void cenv_close() {
    destroy_all();
    g_frame.clear();
}

// Device address of a result buffer of device shard `device_index` (0 .. num_devices - 1): key = "screen" (uint8
// [count * 12288]), "reward" (float [count]), "terminated" / "truncated" (uint8 [count]), "final_screen" (uint8
// [count * 12288], with "final_observation") or "stream" (the cudaStream_t the shard's kernels run on). The same addresses are published as the INT-pair infos "<key>_device". NULL if unknown.
void* cenv_device_buffer(const char* key, int32_t device_index) {
    if (!g_engine || !key || device_index < 0 || (size_t)device_index >= g_engines.size()) return nullptr;
    pg2_engine* e = g_engines[device_index];
    std::string k(key);
    if (k == "screen") return pg2_obs_device(e);
    if (k == "reward") return pg2_reward_device(e);
    if (k == "terminated") return pg2_terminated_device(e);
    if (k == "truncated") return pg2_truncated_device(e);
    if (k == "stream") return pg2_stream(e);
    if (k == "final_screen") return pg2_final_obs_device(e);   // NULL without "final_observation"
    return nullptr;
}

}  // extern "C"
