// Structure-of-arrays game state in HBM. Each game lists its fields once with an X-macro FIELDS(F) of entries
//     F(type, name, elements_per_env)                  scalar `name[env]` or slot-major array `name[i * N + env]`
//                                                      (coalesced across a warp of envs: entity / bullet pools walked
//                                                      by the thread-per-env step kernels)
//     PG2_ENV_MAJOR(F)(type, name, elements_per_env)   env-major array `name[env * K + i]` (contiguous per env: tile
//                                                      maps, which the renderer reads as a window)
// from which the device-visible struct of array pointers, the allocation size and the carving of one big device
// allocation are generated. Both kinds of entry expand alike except in for_each_field, which passes the layout on to
// code that copies one env's elements (the level swap of k_render).
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <string.h>

namespace pg2 {

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

#define PG2_FIELD_DECL(type, name, per_env) type* name;
#define PG2_FIELD_SIZE(type, name, per_env) total += pg2::align256(sizeof(type) * (size_t)(per_env) * (size_t)n);
#define PG2_FIELD_BIND(type, name, per_env) \
    s.name = (type*)(base + off);           \
    off += pg2::align256(sizeof(type) * (size_t)(per_env) * (size_t)n);

#define PG2_FIELD_FIND(type, name, per_env)                                       \
    if (!strcmp(q, #name)) {                                                      \
        *ptr = (void*)this->name; *esz = (int)sizeof(type); *pe = (int)(per_env); \
        return true;                                                              \
    }

#define PG2_FIELD_VISIT(type, name, per_env) fn(#name, (void*)this->name, (int)sizeof(type), (int)(per_env), false);

// An env-major entry names the <generator>_E variant of each generator above.
#define PG2_ENV_MAJOR(F) F##_E
#define PG2_FIELD_DECL_E PG2_FIELD_DECL
#define PG2_FIELD_SIZE_E PG2_FIELD_SIZE
#define PG2_FIELD_BIND_E PG2_FIELD_BIND
#define PG2_FIELD_FIND_E PG2_FIELD_FIND
#define PG2_FIELD_VISIT_E(type, name, per_env) fn(#name, (void*)this->name, (int)sizeof(type), (int)(per_env), true);

#define PG2_DEFINE_STATE(NAME, FIELDS)                                   \
    struct NAME {                                                        \
        int N;                                                           \
        int mode = -1;   /* distribution mode of the level generator (CommonState only; -1: the reference's default) */ \
        FIELDS(PG2_FIELD_DECL)                                           \
        static size_t bytes(int n) {                                     \
            size_t total = 0;                                            \
            FIELDS(PG2_FIELD_SIZE)                                       \
            return total;                                                \
        }                                                                \
        static NAME bind(void* base_, int n) {                           \
            NAME s;                                                      \
            s.N = n;                                                     \
            char* base = (char*)base_;                                   \
            size_t off = 0;                                              \
            FIELDS(PG2_FIELD_BIND)                                       \
            (void)off;                                                   \
            return s;                                                    \
        }                                                                \
        bool find(const char* q, void** ptr, int* esz, int* pe) const {  \
            FIELDS(PG2_FIELD_FIND)                                       \
            return false;                                                \
        }                                                                \
        template <class Fn> void for_each_field(Fn fn) const {           \
            FIELDS(PG2_FIELD_VISIT)                                      \
        }                                                                \
    };

// State every game has (Appendix A of SURVEY.md: what survives reset()).
#define PG2_COMMON_FIELDS(F)                                                                   \
    PG2_ENV_MAJOR(F)(uint32_t, mt, 624) /* std::mt19937 state words */                         \
    F(int32_t, mti, 1)            /* position in the state (624 = twist before next draw) */   \
    F(float, cam_x, 1)            /* gr.camera_position (persists across reset, Q10) */        \
    F(float, cam_y, 1)                                                                         \
    F(uint8_t, sprites_valid, 1)  /* sprite draw list rebuilt since the last reset (Q9) */     \
    F(int32_t, ep_steps, 1)       /* steps in the current episode (max_episode_steps ext.) */  \
    F(int32_t, fault, 1)          /* latent-UB sites of the reference hit (Q20) */                \
    F(uint8_t, view_valid, 1)     /* the env's cached view block (k_render, G::STATIC_VIEW) is current */

PG2_DEFINE_STATE(CommonState, PG2_COMMON_FIELDS)

}  // namespace pg2
