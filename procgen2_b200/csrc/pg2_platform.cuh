// Platform shim. The product is CUDA (sm_100a) only. The PG2_HOSTSIM branch exists solely so
// that tests/hostsim/ can compile these same headers with g++ and single-step the generators
// and the rasteriser against the oracle on the GPU-less build container (fast iteration on
// parity); it is never part of any shipped library and is not a fallback — the engine
// (engine.cu) refuses to start without a CUDA device.
#pragma once
#include <stdint.h>

// engine_final.cu is linked beside engine.cu into one library and includes the same headers: the few non-template,
// non-inline functions they define are static there (it defines PG2_TU_LOCAL as static), so that both translation units
// do not define them. Empty everywhere else.
#ifndef PG2_TU_LOCAL
#define PG2_TU_LOCAL
#endif

#ifndef PG2_HOSTSIM
#include <cuda_runtime.h>
#define PG2_DEV __device__ __forceinline__
#define PG2_DEV_NOINLINE __device__
// A real call (never inlined): large bodies that are reached from several sites (the bit-exact libm restatements, the
// blit axis arithmetic) — one copy keeps the kernels inside the instruction cache.
#define PG2_DEV_CALL __device__ __noinline__
#ifndef PG2_COLD_NOINLINE
#define PG2_COLD_NOINLINE 1
#endif
#if PG2_COLD_NOINLINE
#define PG2_DEV_COLD __device__ __noinline__
#else
#define PG2_DEV_COLD __device__
#endif
namespace pg2 {
constexpr int WARP_LANES = 32;
__device__ __forceinline__ bool warp_any(bool p) { return __any_sync(0xffffffffu, p) != 0; }
__device__ __forceinline__ int warp_sum(int v) { return __reduce_add_sync(0xffffffffu, v); }
__device__ __forceinline__ int warp_bcast(int v) { return __shfl_sync(0xffffffffu, v, 0); }
// the same over a lane group (mask = its lanes; every lane of the group calls with the same mask)
__device__ __forceinline__ bool group_any(uint32_t mask, bool p) { return __any_sync(mask, p) != 0; }
__device__ __forceinline__ int group_sum(uint32_t mask, int v) { return __reduce_add_sync(mask, v); }
__device__ __forceinline__ uint32_t group_or(uint32_t mask, uint32_t v) { return __reduce_or_sync(mask, v); }
__device__ __forceinline__ void group_sync(uint32_t mask) { __syncwarp(mask); }
// atomicAdd on a counter known to live in shared memory (a generic-address atomic costs an address-space dispatch)
__device__ __forceinline__ int smem_atomic_inc(int* p) {
    int old;
    asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(old) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
    return old;
}
__device__ __forceinline__ float warp_bcast(float v) { return __shfl_sync(0xffffffffu, v, 0); }
// Ballot written so that it also works when one thread walks the 32 "virtual lanes" in a loop (host-sim):
// on the GPU the loop body runs once and the result is the ballot; simulated, bit `vlane` is returned and OR-ed up.
__device__ __forceinline__ uint32_t lane_ballot(bool p, int /*vlane*/) { return __ballot_sync(0xffffffffu, p); }
// index of the most significant set bit (0xffffffff for 0)
__device__ __forceinline__ uint32_t bfind(uint32_t v) { uint32_t r; asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(v)); return r; }
__device__ __forceinline__ uint32_t byte_perm(uint32_t a, uint32_t b, uint32_t sel) { return __byte_perm(a, b, sel); }
// Exclusive prefix sum of v over the warp's lanes; *total = the warp's sum. (Host-sim: one lane.)
__device__ __forceinline__ int warp_excl_scan(int v, int* total) {
    const int lane = threadIdx.x & 31;
    int s = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, s, d); if (lane >= d) s += t; }
    *total = __shfl_sync(0xffffffffu, s, 31);
    return s - v;
}
// Lanes of the warp that hold the same key (the caller passes a lane-unique key for "no key").
__device__ __forceinline__ uint32_t match_lanes(uint32_t key) { return __match_any_sync(0xffffffffu, key); }
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t warp_or(uint32_t v) { return __reduce_or_sync(0xffffffffu, v); }
}
#else
#include <math.h>
#include <string.h>
#include <algorithm>
#define PG2_DEV inline
#define PG2_DEV_NOINLINE inline
#define PG2_DEV_CALL inline
#define PG2_DEV_COLD inline
#define __restrict__
namespace pg2 {
constexpr int WARP_LANES = 1;
struct Dim3Sim { int x; };
static const Dim3Sim threadIdx{ 0 }, blockDim{ 1 }, blockIdx{ 0 }, gridDim{ 1 };
inline void __syncthreads() {}
inline void __syncwarp() {}
inline float __fadd_rn(float a, float b) { return a + b; }
inline float __fsub_rn(float a, float b) { return a - b; }
inline float __fmul_rn(float a, float b) { return a * b; }
inline float __fdiv_rn(float a, float b) { return a / b; }
inline float __fsqrt_rn(float a) { return sqrtf(a); }
inline double __dadd_rn(double a, double b) { return a + b; }
inline double __dsub_rn(double a, double b) { return a - b; }
inline double __dmul_rn(double a, double b) { return a * b; }
inline double __ddiv_rn(double a, double b) { return a / b; }
inline float __uint2float_rn(uint32_t u) { return (float)u; }
inline double __fma_rn(double a, double b, double c) { return fma(a, b, c); }
inline uint32_t __float_as_uint(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
inline float __uint_as_float(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
template <class T> inline T __ldg(const T* p) { return *p; }
inline int __ffs(uint32_t m) { return __builtin_ffs((int)m); }
inline int __popc(uint32_t m) { return __builtin_popcount(m); }
inline int __popcll(uint64_t m) { return __builtin_popcountll(m); }
inline int __ffsll(long long m) { return __builtin_ffsll(m); }
inline int __clz(uint32_t m) { return m ? __builtin_clz(m) : 32; }
inline uint32_t __ballot_sync(uint32_t, int pred) { return pred ? 1u : 0u; }
inline bool warp_any(bool p) { return p; }
inline bool group_any(uint32_t, bool p) { return p; }
inline int group_sum(uint32_t, int v) { return v; }
inline uint32_t group_or(uint32_t, uint32_t v) { return v; }
inline void group_sync(uint32_t) {}
inline int warp_sum(int v) { return v; }
inline int warp_bcast(int v) { return v; }
inline float warp_bcast(float v) { return v; }
inline uint32_t atomicOr(uint32_t* p, uint32_t v) { uint32_t o = *p; *p = o | v; return o; }
inline int atomicAdd(int* p, int v) { int o = *p; *p = o + v; return o; }
inline uint32_t atomicExch(uint32_t* p, uint32_t v) { uint32_t o = *p; *p = v; return o; }
inline int smem_atomic_inc(int* p) { return (*p)++; }
inline int atomicMin(int* p, int v) { int o = *p; if (v < o) *p = v; return o; }
inline int atomicMax(int* p, int v) { int o = *p; if (v > o) *p = v; return o; }
inline uint32_t lane_ballot(bool p, int vlane) { return p ? 1u << vlane : 0u; }
inline int warp_excl_scan(int v, int* total) { *total = v; return 0; }
inline uint32_t match_lanes(uint32_t) { return 1u; }
inline int lane_id() { return 0; }
inline uint32_t warp_or(uint32_t v) { return v; }
inline uint32_t bfind(uint32_t v) { return v ? 31u - (uint32_t)__builtin_clz(v) : 0xffffffffu; }
inline uint32_t byte_perm(uint32_t a, uint32_t b, uint32_t sel) {
    uint64_t v = (uint64_t)b << 32 | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) r |= (uint32_t)((v >> (8 * ((sel >> (4 * i)) & 7))) & 255u) << (8 * i);
    return r;
}
using std::max;
using std::min;
}
#endif
