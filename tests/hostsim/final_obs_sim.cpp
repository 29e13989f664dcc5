// TEST INFRASTRUCTURE — NOT PRODUCT CODE, NOT A FALLBACK.
//
// The host-sim (hostsim.cpp, included whole: every hs_* entry point is here too) with the two step variants of the
// engine that the terminal-frame tests (tests/test_hostsim_final_obs.py) compare:
//   auto_reset = 0  a finished env is not reset (pg2_config::auto_reset = 0);
//   final_obs = 1   the terminal frame of a finished env is drawn into its own buffer before the reset
//                   (pg2_config::final_obs).
// The test compiles this file into a temporary directory; nothing under procgen2_b200/ ever loads it.
#include "hostsim.cpp"

struct FinalData {
    bool auto_reset = true, final_on = false;
    std::vector<uint8_t> final_obs;
    virtual ~FinalData() {}
};

template <class G>
struct FinalSim : Sim<G>, FinalData {
    // Sim<G>::step with the two variants
    void step(const int32_t* actions) override {
        for (int e = 0; e < this->N; e++) {
            bool done = step_body<G>(this->st, this->c, e, actions[e], this->reward.data(), this->terminated.data(), this->truncated.data(),
                                     this->max_episode_steps, StepCtx{ 0, 1 });
            if (done && final_on)
                render_body<G>(this->st, this->c, e, *this->frame, this->tex, this->atlas, final_obs.data(),
                               G::STATIC_VIEW ? this->view_cache.data() : nullptr);
            if (done && auto_reset) reset_body<G>(this->st, this->c, e, this->mt_scratch.data(), this->arena.data(), 0);
            this->render(e);
        }
    }
};

extern "C" {

// hs_create_mode with the step variants. final_obs needs auto_reset (like pg2_create): NULL otherwise.
void* hs_create_final(const char* game, int n, int seed, int max_ep, const char* assets, int mode, int auto_reset, int final_obs) {
    if (final_obs && !auto_reset) { g_err = "final_obs needs auto_reset = 1"; return nullptr; }
    std::string g = game;
    if (g_sort_table.empty()) { g_sort_table = build_sort_perm(SORT_MAXN); g_sort_perm = g_sort_table.data(); }
    SimBase* out = nullptr;
    bool ok = false;
#define PG2_FINAL_SIM(TYPE)                                                                                  \
    {                                                                                                        \
        auto* s = new FinalSim<TYPE>();                                                                      \
        out = s;                                                                                             \
        ok = s->init(n, (uint32_t)seed, max_ep, assets, &g_err, mode);                                       \
        s->auto_reset = auto_reset != 0; s->final_on = final_obs != 0; s->final_obs.assign((size_t)n * OBS_BYTES, 0); \
    }
#define PG2_TRY_GAME_MODE(NAME, MODE, TYPE) if (!out && g == NAME && mode == MODE) PG2_FINAL_SIM(TYPE)
    PG2_FOR_EACH_GAME_MODE(PG2_TRY_GAME_MODE)
#undef PG2_TRY_GAME_MODE
#define PG2_TRY_GAME(NAME, TYPE) if (!out && g == NAME) PG2_FINAL_SIM(TYPE)
    PG2_FOR_EACH_GAME(PG2_TRY_GAME)
#undef PG2_TRY_GAME
#undef PG2_FINAL_SIM
    if (!out) { g_err = "unknown game " + g; return nullptr; }
    if (!ok) { delete out; return nullptr; }
    return out;
}

// The terminal frames of a sim made by hs_create_final: N * 12288 bytes, row e written in the steps env e finished in.
// NULL for a sim made by hs_create / hs_create_mode.
const uint8_t* hs_final_obs(void* h) {
    FinalData* f = dynamic_cast<FinalData*>((SimBase*)h);
    return f ? f->final_obs.data() : nullptr;
}

}  // extern "C"
