// TEST INFRASTRUCTURE. Draws synthetic scenes (scene.h) with the production rasteriser, for tests/test_raster_spec.py.
// One source, two builds (tests/raster/build.py):
//   nvcc (sm_100a, the engine's flags)   the production kernels k_render / k_render_human (pg2_kernels.cuh) instantiated
//                                        for SynthOf<G>: persistent CTAs, frame tickets, TMA bulk stores, view cache
//   g++ -DPG2_HOSTSIM                    render_body / render_human_body run by one host thread (as tests/hostsim/), which
//                                        also reports the rasteriser's slow-path counters
// Per frame the report holds (SC_REPORT_OUT words): 0 wide, 1 npost, 2 reuse, 3 overflow, 4 fault; host build only:
// 5 g_dbg_slow, 6 g_dbg_quads, 7 g_dbg_quads_slow, 8 g_dbg_rb, 9 RC_AMBIGUOUS rowcell entries, 10 rotated post blits,
// 11 pre_blend (the background has alpha), 12 screen rows + columns the background leaves uncovered.
// The GPU build draws the same scenes from the same source; the tests take path coverage from the host build's report.
#include <stdio.h>
#include <string.h>
#include <memory>
#include <vector>

#include "../../procgen2_b200/csrc/games/all_games.cuh"
#include "synth_game.cuh"

using namespace pg2;

#define SC_REPORT_OUT 13

// The trait sets tested, by index (the games' render traits; chaser mode 2 has the largest post-blit list).
#define PG2_FOR_EACH_TRAIT(X) \
    X(0, pg2::Maze)           \
    X(1, pg2::CoinRun)        \
    X(2, pg2::Climber)        \
    X(3, pg2::Jumper)         \
    X(4, pg2::BossFight)      \
    X(5, pg2::CaveFlyer)      \
    X(6, pg2::ChaserT<2>)

static bool base_changed(const sc_scene& a, const sc_scene& b) {
    return memcmp(&a, &b, SC_BASE_BYTES) != 0 || memcmp(a.map, b.map, sizeof(a.map)) != 0;
}

#ifndef PG2_HOSTSIM
#define RH_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { fprintf(stderr, "%s: %s\n", #call, cudaGetErrorString(e__)); return -1; } } while (0)

struct DevBufs {
    std::vector<void*> ptrs;
    ~DevBufs() { for (void* p : ptrs) cudaFree(p); }
    template <class T> T* alloc(size_t bytes) { void* p = nullptr; if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr; ptrs.push_back(p); cudaMemset(p, 0, bytes); return (T*)p; }
};

// npass x nenv scenes: pass p draws every env once (one k_render launch); an env whose base image (camera, background,
// tile map) is the same as in the previous pass keeps its cached view, as in an episode of a STATIC_VIEW game.
template <class G>
static int run_frames(int npass, int nenv, const sc_scene* scenes, const TexInfo* tex_h, int ntex, const uint32_t* atlas_h, long natlas,
                      int grid, uint8_t* obs_out, int32_t* report_out) {
    using S = SynthOf<G>;
    DevBufs d;
    char* smem = d.alloc<char>(SynthState::bytes(nenv));
    char* cmem = d.alloc<char>(CommonState::bytes(nenv));
    TexInfo* tex = d.alloc<TexInfo>(sizeof(TexInfo) * ntex);
    uint32_t* atlas = d.alloc<uint32_t>(sizeof(uint32_t) * natlas);
    uint8_t* obs = d.alloc<uint8_t>((size_t)nenv * OBS_BYTES);
    uint8_t* cache = d.alloc<uint8_t>((size_t)nenv * VIEW_CACHE_BYTES);
    int* ticket = d.alloc<int>(sizeof(int));
    if (!smem || !cmem || !tex || !atlas || !obs || !cache || !ticket) return -1;
    SynthState s = SynthState::bind(smem, nenv);
    CommonState c = CommonState::bind(cmem, nenv);
    RH_CUDA(cudaMemcpy(tex, tex_h, sizeof(TexInfo) * ntex, cudaMemcpyHostToDevice));
    RH_CUDA(cudaMemcpy(atlas, atlas_h, sizeof(uint32_t) * natlas, cudaMemcpyHostToDevice));
    if (grid <= 0) {
        int per_sm = 0, dev = 0, sms = 0;
        RH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_render<S, false>, RENDER_THREADS, 0));
        RH_CUDA(cudaGetDevice(&dev));
        RH_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        grid = nenv < sms * per_sm ? nenv : sms * per_sm;
    }
    SwapArgs swap;
    memset(&swap, 0, sizeof(swap));
    std::vector<uint8_t> valid(nenv);
    std::vector<int32_t> rep((size_t)nenv * SC_REPORT), fault(nenv);
    for (int p = 0; p < npass; p++) {
        const sc_scene* sp = scenes + (size_t)p * nenv;
        RH_CUDA(cudaMemcpy(s.scene, sp, sizeof(sc_scene) * nenv, cudaMemcpyHostToDevice));
        RH_CUDA(cudaMemcpy(valid.data(), c.view_valid, nenv, cudaMemcpyDeviceToHost));
        for (int e = 0; e < nenv; e++) if (p == 0 || base_changed(sp[e], sp[e - nenv])) valid[e] = 0;
        RH_CUDA(cudaMemcpy(c.view_valid, valid.data(), nenv, cudaMemcpyHostToDevice));
        RH_CUDA(cudaMemset(c.fault, 0, sizeof(int32_t) * nenv));
        RH_CUDA(cudaMemset(ticket, 0, sizeof(int)));
        k_render<S, false><<<grid, RENDER_THREADS>>>(s, c, tex, atlas, obs, ticket, 0, nullptr, nullptr, nullptr, nenv, cache, swap, nullptr, nullptr);
        RH_CUDA(cudaGetLastError());
        RH_CUDA(cudaDeviceSynchronize());
        RH_CUDA(cudaMemcpy(obs_out + (size_t)p * nenv * OBS_BYTES, obs, (size_t)nenv * OBS_BYTES, cudaMemcpyDeviceToHost));
        RH_CUDA(cudaMemcpy(rep.data(), s.report, sizeof(int32_t) * SC_REPORT * nenv, cudaMemcpyDeviceToHost));
        RH_CUDA(cudaMemcpy(fault.data(), c.fault, sizeof(int32_t) * nenv, cudaMemcpyDeviceToHost));
        for (int e = 0; e < nenv; e++) {
            int32_t* r = report_out + ((size_t)p * nenv + e) * SC_REPORT_OUT;
            r[0] = rep[e * SC_REPORT]; r[1] = rep[e * SC_REPORT + 1]; r[2] = rep[e * SC_REPORT + 2];
            r[3] = (fault[e] & 8) ? 1 : 0; r[4] = fault[e];
        }
    }
    return 0;
}

// One human-mode frame (render_game(false) at width x height), drawn by `grid` CTAs (k_render_human).
template <class G>
static int run_human(const sc_scene* scene, const TexInfo* tex_h, int ntex, const uint32_t* atlas_h, long natlas,
                     int width, int height, int grid, uint8_t* out_h, int32_t* report_out) {
    using S = SynthOf<G>;
    DevBufs d;
    char* smem = d.alloc<char>(SynthState::bytes(1));
    char* cmem = d.alloc<char>(CommonState::bytes(1));
    TexInfo* tex = d.alloc<TexInfo>(sizeof(TexInfo) * ntex);
    uint32_t* atlas = d.alloc<uint32_t>(sizeof(uint32_t) * natlas);
    uint8_t* out = d.alloc<uint8_t>((size_t)width * height * 3);
    int* overflow = d.alloc<int>(sizeof(int));
    if (!smem || !cmem || !tex || !atlas || !out || !overflow) return -1;
    SynthState s = SynthState::bind(smem, 1);
    CommonState c = CommonState::bind(cmem, 1);
    RH_CUDA(cudaMemcpy(s.scene, scene, sizeof(sc_scene), cudaMemcpyHostToDevice));
    RH_CUDA(cudaMemcpy(tex, tex_h, sizeof(TexInfo) * ntex, cudaMemcpyHostToDevice));
    RH_CUDA(cudaMemcpy(atlas, atlas_h, sizeof(uint32_t) * natlas, cudaMemcpyHostToDevice));
    k_render_human<S><<<grid, RENDER_THREADS>>>(s, c, 0, tex, atlas, out, width, height, overflow);
    RH_CUDA(cudaGetLastError());
    RH_CUDA(cudaDeviceSynchronize());
    RH_CUDA(cudaMemcpy(out_h, out, (size_t)width * height * 3, cudaMemcpyDeviceToHost));
    int32_t rep[SC_REPORT], ov = 0;
    RH_CUDA(cudaMemcpy(rep, s.report, sizeof(rep), cudaMemcpyDeviceToHost));
    RH_CUDA(cudaMemcpy(&ov, overflow, sizeof(int), cudaMemcpyDeviceToHost));
    report_out[0] = rep[0]; report_out[1] = rep[1]; report_out[2] = rep[2]; report_out[3] = ov; report_out[4] = 0;
    return 0;
}
#else
static void dbg_report(int32_t* r, const long* before) {
    r[5] = (int32_t)(g_dbg_slow - before[0]); r[6] = (int32_t)(g_dbg_quads - before[1]);
    r[7] = (int32_t)(g_dbg_quads_slow - before[2]); r[8] = (int32_t)(g_dbg_rb - before[3]);
}

template <class G>
static int run_frames(int npass, int nenv, const sc_scene* scenes, const TexInfo* tex, int, const uint32_t* atlas, long,
                      int, uint8_t* obs_out, int32_t* report_out) {
    using S = SynthOf<G>;
    std::vector<char> smem(SynthState::bytes(nenv)), cmem(CommonState::bytes(nenv));
    std::vector<uint8_t> cache((size_t)nenv * VIEW_CACHE_BYTES);
    SynthState s = SynthState::bind(smem.data(), nenv);
    CommonState c = CommonState::bind(cmem.data(), nenv);
    std::unique_ptr<FrameOf<S>> f(new FrameOf<S>());
    frame_init_tiletex<S>(*f, tex);
    for (int p = 0; p < npass; p++) {
        const sc_scene* sp = scenes + (size_t)p * nenv;
        memcpy(s.scene, sp, sizeof(sc_scene) * nenv);
        for (int e = 0; e < nenv; e++) {
            if (p == 0 || base_changed(sp[e], sp[e - nenv])) c.view_valid[e] = 0;
            c.fault[e] = 0;
            const long before[4] = { g_dbg_slow, g_dbg_quads, g_dbg_quads_slow, g_dbg_rb };
            render_body<S>(s, c, e, *f, tex, atlas, obs_out + (size_t)p * nenv * OBS_BYTES, S::STATIC_VIEW ? cache.data() : nullptr);
            int32_t* r = report_out + ((size_t)p * nenv + e) * SC_REPORT_OUT;
            r[0] = f->wide; r[1] = f->npost; r[2] = f->reuse; r[3] = (c.fault[e] & 8) ? 1 : 0; r[4] = c.fault[e];
            dbg_report(r, before);
            int amb = 0;
            if (!f->reuse && !f->wide)
                for (int k = 0; k < f->nrow * OBS_W; k++) amb += (f->rowcell[k] & RC_AMBIGUOUS) != 0u;
            r[9] = amb;
            int nrot = 0, holes = 0;
            for (int k = 0; k < f->npost; k++) nrot += (f->fpost[k].flags & 2u) != 0u;
            if (!f->reuse && !f->wide)
                for (int k = 0; k < OBS_W; k++) holes += (f->rowf[k].pre_row == (int32_t)BG_HOLE) + (f->col_pre[k] < 0);
            r[10] = nrot; r[11] = f->reuse ? 0 : f->pre_blend; r[12] = holes;
        }
    }
    return 0;
}

template <class G>
static int run_human(const sc_scene* scene, const TexInfo* tex, int, const uint32_t* atlas, long,
                     int width, int height, int, uint8_t* out, int32_t* report_out) {
    using S = SynthOf<G>;
    std::vector<char> smem(SynthState::bytes(1)), cmem(CommonState::bytes(1));
    SynthState s = SynthState::bind(smem.data(), 1);
    CommonState c = CommonState::bind(cmem.data(), 1);
    memcpy(s.scene, scene, sizeof(sc_scene));
    std::unique_ptr<FrameOf<S>> f(new FrameOf<S>());
    frame_init_tiletex<S>(*f, tex);
    const long before[4] = { g_dbg_slow, g_dbg_quads, g_dbg_quads_slow, g_dbg_rb };
    const bool ok = render_human_body<S>(s, c, 0, *f, tex, atlas, out, width, height, 0, width * height);
    report_out[0] = f->wide; report_out[1] = f->npost; report_out[2] = f->reuse; report_out[3] = ok ? 0 : 1; report_out[4] = 0;
    dbg_report(report_out, before);
    report_out[9] = 0;
    int nrot = 0;
    for (int k = 0; k < f->npost; k++) nrot += (f->fpost[k].flags & 2u) != 0u;
    report_out[10] = nrot; report_out[11] = f->pre_blend; report_out[12] = 0;
    return 0;
}
#endif

// exported from the nvcc build too, which compiles with -fvisibility=hidden
#define RH_API __attribute__((visibility("default")))

extern "C" {

RH_API int rh_report_words() { return SC_REPORT_OUT; }
RH_API int rh_scene_bytes() { return (int)sizeof(sc_scene); }
RH_API int rh_is_gpu() {
#ifdef PG2_HOSTSIM
    return 0;
#else
    return 1;
#endif
}

// scenes: [npass][nenv]; obs_out: [npass][nenv][64][64][3]; report_out: [npass][nenv][SC_REPORT_OUT].
// grid: CTAs of each k_render launch (<= 0: the occupancy-sized grid the engine uses). Returns 0, or -1 on an error.
RH_API int rh_render(int trait, int npass, int nenv, const sc_scene* scenes, const TexInfo* tex, int ntex, const uint32_t* atlas, long natlas,
              int grid, uint8_t* obs_out, int32_t* report_out) {
    if (ntex < SC_NUM_TEX) return -1;
#define PG2_TRAIT_CASE(k, T) if (trait == k) return run_frames<T>(npass, nenv, scenes, tex, ntex, atlas, natlas, grid, obs_out, report_out);
    PG2_FOR_EACH_TRAIT(PG2_TRAIT_CASE)
#undef PG2_TRAIT_CASE
    return -1;
}

// out: [height][width][3]; report_out: SC_REPORT_OUT words (overflow: the frame is incomplete, render_human_body).
RH_API int rh_render_human(int trait, const sc_scene* scene, const TexInfo* tex, int ntex, const uint32_t* atlas, long natlas,
                    int width, int height, int grid, uint8_t* out, int32_t* report_out) {
    if (ntex < SC_NUM_TEX || width < 1 || height < 1 || grid < 1) return -1;
#define PG2_TRAIT_CASE(k, T) if (trait == k) return run_human<T>(scene, tex, ntex, atlas, natlas, width, height, grid, out, report_out);
    PG2_FOR_EACH_TRAIT(PG2_TRAIT_CASE)
#undef PG2_TRAIT_CASE
    return -1;
}

}  // extern "C"
