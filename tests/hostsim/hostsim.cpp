// TEST INFRASTRUCTURE — NOT PRODUCT CODE, NOT A FALLBACK.
//
// Single-threaded host build of the engine's device headers (PG2_HOSTSIM, see
// procgen2_b200/csrc/pg2_platform.cuh): lets the CPU-only test-suite step the very same
// generator / step / rasteriser source against the oracle (oracle/_ref) with a seconds-long
// edit-compile-run loop, before the result is confirmed on a B200 by the `-m gpu` tests.
// Built by tests/hostsim/build.py into tests/hostsim/_build/libpg2_hostsim.so; nothing under
// procgen2_b200/ ever loads it.
#define PG2_HOSTSIM 1
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../procgen2_b200/csrc/assets.h"
#include "../../procgen2_b200/csrc/games/all_games.cuh"
#include "../../procgen2_b200/csrc/pg2_kernels.cuh"
#include "../../procgen2_b200/csrc/sort_perm.h"

using namespace pg2;

struct SimBase {
    virtual ~SimBase() {}
    virtual void reset_all(const int32_t* seeds) = 0;
    virtual void step(const int32_t* actions) = 0;
    virtual bool find_field(const char* name, void** ptr, int* esz, int* pe) = 0;
    virtual bool render_human(int env, int width, int height, uint8_t* out) = 0;
    virtual void invalidate_views() = 0;
    // every field of the game state, then of CommonState, in declaration order (for_each_field)
    struct FieldInfo { std::string name; void* ptr; int esz, per_env; bool env_major; };
    std::vector<FieldInfo> fields;
    int N = 0, max_episode_steps = 0;
    // the engine's step variants: auto_reset = false (pg2_config::auto_reset = 0) does not reset a finished env; final_on
    // (pg2_config::final_obs) draws the terminal frame of a finished env into final_obs before the reset
    bool auto_reset = true, final_on = false;
    std::vector<uint8_t> obs, terminated, truncated, final_obs;
    std::vector<float> reward;
};

template <class G>
struct Sim : SimBase {
    typename G::State st;
    CommonState c;
    std::vector<char> state_mem, common_mem, arena;
    std::vector<uint8_t> view_cache;
    std::vector<uint32_t> mt_scratch;
    const TexInfo* tex = nullptr;
    const uint32_t* atlas = nullptr;
    std::unique_ptr<FrameOf<G>> frame;

    bool init(int n, uint32_t base_seed, int max_ep, const char* assets, std::string* err, int mode = -1) {
        N = n; max_episode_steps = max_ep;
        state_mem.assign(G::State::bytes(N), 0);
        common_mem.assign(CommonState::bytes(N), 0);
        st = G::State::bind(state_mem.data(), N);
        c = CommonState::bind(common_mem.data(), N);
        c.mode = mode;
        arena.assign(G::RESET_ARENA, 0);
        view_cache.assign((size_t)N * VIEW_CACHE_BYTES, 0);
        mt_scratch.assign(MT_N, 0);
        frame.reset(new FrameOf<G>());
        obs.assign((size_t)N * OBS_BYTES, 0); terminated.assign(N, 0); truncated.assign(N, 0); reward.assign(N, 0.0f);
        int ntex = 0;
        const char* const* names = G::texture_names(&ntex);
        // decoding the textures dominates creation, and the parity tests create thousands of one-env sims
        static std::map<std::pair<std::string, const char* const*>, std::pair<std::vector<TexInfo>, std::vector<uint32_t>>> loaded;
        auto key = std::make_pair(std::string(assets ? assets : ""), names);
        auto it = loaded.find(key);
        if (it == loaded.end()) {
            std::vector<TexInfo> t;
            std::vector<uint32_t> a;
            if (!load_textures(assets, names, ntex, &t, &a, err)) return false;
            it = loaded.emplace(key, std::make_pair(std::move(t), std::move(a))).first;
        }
        tex = it->second.first.data();
        atlas = it->second.second.data();
        frame_init_tiletex<G>(*frame, tex);
        auto add = [&](const char* name, void* p, int esz, int pe, bool em) { fields.push_back(FieldInfo{ name, p, esz, pe, em }); };
        st.for_each_field(add);
        c.for_each_field(add);
        for (int e = 0; e < N; e++) seed_body(c, e, base_seed + (uint32_t)e, true);
        for (int e = 0; e < N; e++) reset_body<G>(st, c, e, mt_scratch.data(), arena.data(), 0);
        return true;
    }
    void render(int e) { render_body<G>(st, c, e, *frame, tex, atlas, obs.data(), G::STATIC_VIEW ? view_cache.data() : nullptr); }
    void reset_all(const int32_t* seeds) override {
        for (int e = 0; e < N; e++) {
            if (seeds) seed_body(c, e, (uint32_t)seeds[e], false);
            reset_body<G>(st, c, e, mt_scratch.data(), arena.data(), 0);
            render(e);
            reward[e] = 0.0f; terminated[e] = 0; truncated[e] = 0;
        }
    }
    void step(const int32_t* actions) override {
        for (int e = 0; e < N; e++) {
            bool done = step_body<G>(st, c, e, actions[e], reward.data(), terminated.data(), truncated.data(), max_episode_steps, StepCtx{ 0, 1 });
            if (done && final_on) render_body<G>(st, c, e, *frame, tex, atlas, final_obs.data(), G::STATIC_VIEW ? view_cache.data() : nullptr);
            if (done && auto_reset) reset_body<G>(st, c, e, mt_scratch.data(), arena.data(), 0);
            render(e);
        }
    }
    bool find_field(const char* name, void** ptr, int* esz, int* pe) override {
        return st.find(name, ptr, esz, pe) || c.find(name, ptr, esz, pe);
    }
    bool render_human(int env, int width, int height, uint8_t* out) override {
        return render_human_body<G>(st, c, env, *frame, tex, atlas, out, width, height, 0, width * height);
    }
    // the view cache is this sim's own: state copied in from elsewhere says nothing about it
    void invalidate_views() override { memset(c.view_valid, 0, (size_t)N); }
};

static std::string g_err;
static std::vector<uint8_t> g_sort_table;

extern "C" {

const char* hs_last_error() { return g_err.c_str(); }
void hs_debug_counters(long* out) { out[0] = pg2::g_dbg_slow; out[1] = pg2::g_dbg_quads; out[2] = pg2::g_dbg_quads_slow; out[3] = pg2::g_dbg_rb; }

// mode: the distribution mode (-1: the game's default). auto_reset / final_obs: the step variants (SimBase); final_obs
// needs auto_reset (like pg2_create): NULL otherwise.
void* hs_create(const char* game, int n, int seed, int max_ep, const char* assets, int mode, int auto_reset, int final_obs) {
    if (final_obs && !auto_reset) { g_err = "final_obs needs auto_reset = 1"; return nullptr; }
    std::string g = game;
    if (g_sort_table.empty()) { g_sort_table = build_sort_perm(SORT_MAXN); g_sort_perm = g_sort_table.data(); }
    SimBase* out = nullptr;
    bool ok = false;
#define PG2_TRY_GAME_MODE(NAME, MODE, TYPE) \
    if (!out && g == NAME && mode == MODE) { auto* s = new Sim<TYPE>(); out = s; ok = s->init(n, (uint32_t)seed, max_ep, assets, &g_err, mode); }
    PG2_FOR_EACH_GAME_MODE(PG2_TRY_GAME_MODE)
#undef PG2_TRY_GAME_MODE
#define PG2_TRY_GAME(NAME, TYPE) \
    if (!out && g == NAME) { auto* s = new Sim<TYPE>(); out = s; ok = s->init(n, (uint32_t)seed, max_ep, assets, &g_err, mode); }
    PG2_FOR_EACH_GAME(PG2_TRY_GAME)
#undef PG2_TRY_GAME
    if (!out) { g_err = "unknown game " + g; return nullptr; }
    if (!ok) { delete out; return nullptr; }
    out->auto_reset = auto_reset != 0;
    out->final_on = final_obs != 0;
    if (out->final_on) out->final_obs.assign((size_t)n * OBS_BYTES, 0);
    return out;
}
void hs_destroy(void* h) { delete (SimBase*)h; }
void hs_reset(void* h, const int32_t* seeds) { ((SimBase*)h)->reset_all(seeds); }
void hs_step(void* h, const int32_t* actions) { ((SimBase*)h)->step(actions); }
// 0: done; 1: the window spans more tile rows than the frame tables hold (the engine's pg2_render_human fails)
int hs_render_human(void* h, int env, int width, int height, uint8_t* out) { return ((SimBase*)h)->render_human(env, width, height, out) ? 0 : 1; }
const uint8_t* hs_obs(void* h) { return ((SimBase*)h)->obs.data(); }
const float* hs_reward(void* h) { return ((SimBase*)h)->reward.data(); }
const uint8_t* hs_terminated(void* h) { return ((SimBase*)h)->terminated.data(); }
const uint8_t* hs_truncated(void* h) { return ((SimBase*)h)->truncated.data(); }
// The terminal frames of a sim created with final_obs: N * 12288 bytes, row e written in the steps env e finished in.
// NULL for a sim without final_obs.
const uint8_t* hs_final_obs(void* h) { SimBase* s = (SimBase*)h; return s->final_on ? s->final_obs.data() : nullptr; }
long hs_read_field(void* h, const char* name, void* out, long capacity, int* elem_size, int* per_env) {
    SimBase* s = (SimBase*)h;
    void* ptr; int esz, pe;
    if (!s->find_field(name, &ptr, &esz, &pe)) return -1;
    if (elem_size) *elem_size = esz;
    if (per_env) *per_env = pe;
    long bytes = (long)esz * pe * s->N;
    if (!out) return bytes;
    if (capacity < bytes) return -2;
    memcpy(out, ptr, bytes);
    return bytes;
}
// Counterpart of hs_read_field: `bytes` must be the field's whole size. Returns it, -1: unknown field, -2: size mismatch.
long hs_write_field(void* h, const char* name, const void* in, long bytes) {
    SimBase* s = (SimBase*)h;
    void* ptr; int esz, pe;
    if (!s->find_field(name, &ptr, &esz, &pe)) return -1;
    if (bytes != (long)esz * pe * s->N) return -2;
    memcpy(ptr, in, bytes);
    return bytes;
}
int hs_field_count(void* h) { return (int)((SimBase*)h)->fields.size(); }
// Field i of hs_field_count: its name (copied into name_out, 64 bytes), element size, elements per env and layout
// (1: env-major `name[env * per_env + k]`, 0: `name[k * N + env]`). Returns 0, or -1 for an index out of range.
int hs_field_info(void* h, int i, char* name_out, int* esz, int* per_env, int* env_major) {
    SimBase* s = (SimBase*)h;
    if (i < 0 || i >= (int)s->fields.size()) return -1;
    const SimBase::FieldInfo& f = s->fields[i];
    snprintf(name_out, 64, "%s", f.name.c_str());
    *esz = f.esz; *per_env = f.per_env; *env_major = f.env_major ? 1 : 0;
    return 0;
}
void hs_invalidate_views(void* h) { ((SimBase*)h)->invalidate_views(); }

}  // extern "C"
