// Device restatement of the reference's random stream: one std::mt19937 per environment
// (games/coinrun/coinrun.cpp:34 `std::mt19937 rng;`, seeded `rng.seed(seed)` coinrun.cpp:235)
// consumed through libstdc++ 13 distributions:
//   std::uniform_int_distribution<int>   -> Lemire nearly-divisionless (bits/uniform_int_dist.h:257-279,305-328)
//   std::uniform_real_distribution<float> -> generate_canonical<float,24> (bits/random.tcc:3349-3380)
// so that a given seed yields the identical level (SURVEY Q1-Q3).
#pragma once
#include <stdint.h>
#include "pg2_platform.cuh"

namespace pg2 {

constexpr int MT_N = 624;
constexpr int MT_M = 397;

// Generator view: `mt` points at 624 state words (shared or global memory), `idx` is the
// position kept in a register by the caller and written back when done.
struct Mt {
    uint32_t* mt;
    int idx;
    // warp-per-env step kernels run the generator redundantly on all 32 lanes (identical idx): `collective` makes the
    // in-place twist of the shared global state a one-lane job (`writer`) followed by a warp barrier
    bool collective = false, writer = true;
    uint32_t sync_mask = 0xffffffffu;   // the lanes that run this generator together

    PG2_DEV static uint32_t mix(uint32_t u, uint32_t v, uint32_t m) {
        uint32_t y = (u & 0x80000000u) | (v & 0x7fffffffu);
        return m ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }

    // single-thread twist (thread-per-env kernels)
    PG2_DEV_CALL void twist_serial() {
        for (int k = 0; k < MT_N - MT_M; k++) mt[k] = mix(mt[k], mt[k + 1], mt[k + MT_M]);
        for (int k = MT_N - MT_M; k < MT_N - 1; k++) mt[k] = mix(mt[k], mt[k + 1], mt[k + (MT_M - MT_N)]);
        mt[MT_N - 1] = mix(mt[MT_N - 1], mt[0], mt[MT_M - 1]);
        idx = 0;
    }

    PG2_DEV uint32_t next() {
        if (idx >= MT_N) {
            if (!collective) twist_serial();
            else { if (writer) twist_serial(); idx = 0; group_sync(sync_mask); }
        }
        uint32_t y = mt[idx++];
        y ^= (y >> 11);
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= (y >> 18);
        return y;
    }

    // uniform_int_distribution<int>(a, b)(rng): always consumes >= 1 draw, even for a == b.
    PG2_DEV int uniform_int(int a, int b) {
        uint32_t urange = (uint32_t)b - (uint32_t)a;
        if (urange == 0xffffffffu) return (int)(next() + (uint32_t)a);
        uint32_t uerange = urange + 1u;
        uint64_t product = (uint64_t)next() * (uint64_t)uerange;
        uint32_t low = (uint32_t)product;
        if (low < uerange) {
            uint32_t threshold = (0u - uerange) % uerange;
            while (low < threshold) {
                product = (uint64_t)next() * (uint64_t)uerange;
                low = (uint32_t)product;
            }
        }
        return (int)((uint32_t)(product >> 32) + (uint32_t)a);
    }

    // uniform_real_distribution<float>(0,1)(rng): one draw; float(u32) rounds to nearest,
    // a result of 1.0f is clamped to nextafterf(1, 0).
    PG2_DEV float canonical() {
        float r = __fdiv_rn(__uint2float_rn(next()), 4294967296.0f);
        if (r >= 1.0f) r = 0.99999994f;
        return r;
    }
    PG2_DEV float uniform_real(float a, float b) {
        return __fadd_rn(__fmul_rn(canonical(), __fsub_rn(b, a)), a);
    }
};

// Warp-collective generator used by the level-generation kernel: the 624 state words sit in
// shared memory, all 32 lanes execute the (uniform) generator code redundantly and therefore
// hold identical `idx`; the twist — the only bulk work — is spread over the lanes.
struct WarpMt {
    uint32_t* mt;   // shared memory, 624 words
    int idx;
    int lane;

    PG2_DEV_CALL void twist() {
        __syncwarp();
        // new[k] = mix(mt[k], mt[k+1 mod N], mt[k+M mod N]) in ascending k; chunks of 32 read
        // their inputs before any lane of the chunk writes, later chunks see the updated words
        // exactly as the serial algorithm does (k+1 is still old, k+M-N (k >= N-M) is new).
        for (int base = 0; base < MT_N; base += WARP_LANES) {
            int k = base + lane;
            uint32_t v = 0;
            if (k < MT_N) {
                int k1 = (k + 1 == MT_N) ? 0 : k + 1;
                int km = (k + MT_M >= MT_N) ? k + MT_M - MT_N : k + MT_M;
                v = Mt::mix(mt[k], mt[k1], mt[km]);
            }
            __syncwarp();
            if (k < MT_N) mt[k] = v;
            __syncwarp();
        }
        idx = 0;
    }

    // n consecutive uniform_real_distribution<float>(0,1) draws compared against per-draw thresholds, spread over the
    // lanes: out[i] = draw_i < thr(i). Identical stream consumption to n calls of canonical() (one word per draw).
    template <class Thr>
    PG2_DEV_NOINLINE void bernoulli_fill(uint8_t* out, int n, Thr thr) {
        int done = 0;
        while (done < n) {
            if (idx >= MT_N) twist();
            int m = min(MT_N - idx, n - done);
            __syncwarp();
            for (int j = lane; j < m; j += WARP_LANES) {
                uint32_t y = mt[idx + j];
                y ^= (y >> 11);
                y ^= (y << 7) & 0x9d2c5680u;
                y ^= (y << 15) & 0xefc60000u;
                y ^= (y >> 18);
                float r = __fdiv_rn(__uint2float_rn(y), 4294967296.0f);
                if (r >= 1.0f) r = 0.99999994f;
                out[done + j] = r < thr(done + j) ? 1 : 0;
            }
            __syncwarp();
            idx += m; done += m;
        }
    }

    PG2_DEV uint32_t next() {
        if (idx >= MT_N) twist();
        uint32_t y = mt[idx++];
        y ^= (y >> 11);
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= (y >> 18);
        return y;
    }
    PG2_DEV int uniform_int(int a, int b) {
        uint32_t urange = (uint32_t)b - (uint32_t)a;
        if (urange == 0xffffffffu) return (int)(next() + (uint32_t)a);
        uint32_t uerange = urange + 1u;
        uint64_t product = (uint64_t)next() * (uint64_t)uerange;
        uint32_t low = (uint32_t)product;
        if (low < uerange) {
            uint32_t threshold = (0u - uerange) % uerange;
            while (low < threshold) {
                product = (uint64_t)next() * (uint64_t)uerange;
                low = (uint32_t)product;
            }
        }
        return (int)((uint32_t)(product >> 32) + (uint32_t)a);
    }
    PG2_DEV float canonical() {
        float r = __fdiv_rn(__uint2float_rn(next()), 4294967296.0f);
        if (r >= 1.0f) r = 0.99999994f;
        return r;
    }
    PG2_DEV float uniform_real(float a, float b) {
        return __fadd_rn(__fmul_rn(canonical(), __fsub_rn(b, a)), a);
    }
};

// rng.seed(seed): mt[0] = seed; mt[i] = 1812433253 * (mt[i-1] ^ (mt[i-1] >> 30)) + i; position = 624.
PG2_TU_LOCAL PG2_DEV_NOINLINE void mt_seed(uint32_t* mt, uint32_t seed) {
    uint32_t x = seed;
    mt[0] = x;
    for (int i = 1; i < MT_N; i++) {
        x = 1812433253u * (x ^ (x >> 30)) + (uint32_t)i;
        mt[i] = x;
    }
}

}  // namespace pg2
