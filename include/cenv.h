/* procgen2-b200 — the `cenv` environment ABI this project is a drop-in for.
 *
 * This header declares, in this project's own words, the binary interface defined by the
 * reference at /root/reference/cenv/cenv.h:26-133 (six entry points + four exported result
 * structs) and consumed by its ctypes wrapper cenv/cenv.py:62-111, 160-182. Names, field order,
 * field types and enum values are the contract and therefore identical; layout facts on LP64:
 *   cenv_key_value 24 B {key@0, value_type@8, value_buffer_size@12, value_buffer@16}
 *   cenv_option    24 B {name@0, value_type@8, value@16}
 *   cenv_step_data 40 B {observations_size@0, observations@8, reward@16, terminated@24,
 *                        truncated@25, infos_size@28, infos@32}
 * (static_asserts in procgen2_b200/csrc/cenv_abi.cpp pin them).
 *
 * Batched extension implemented by this project's libraries (reference: one env per library):
 *   make options  "num_envs" (INT, default 1), "device" (INT, default 0),
 *                 "num_devices" (INT, default 1: devices device .. device + num_devices - 1 each own a
 *                 contiguous slice of the envs; env i is seeded seed + i whatever the device count),
 *                 "max_episode_steps" (INT, default 0 = never truncate),
 *                 "auto_reset" (INT, default 1 when num_envs > 1, else 0),
 *                 "distribution_mode" (INT, default -1 = the mode the reference compiles in; 0 easy, 1 hard, 2 memory /
 *                 extreme — games/<g>/tilemap.h Config, bossfight common_systems.h:44-65; every mode a game has is built,
 *                 one it does not have makes cenv_make fail),
 *                 "host_copy" (INT, default 1; 0: observations stay device-resident — cenv_step / cenv_reset return
 *                 when the kernels have finished, without the device -> host copy of "screen"; rewards and flags are
 *                 still copied),
 *                 "final_observation" (INT, default 0; auto-reset only, cenv_make fails with auto_reset 0: there the
 *                 "screen" of a finished env already is its terminal frame): also return the frame each finished
 *                 episode ended in, which auto-reset replaces in "screen" by the first frame of the next episode
 *   actions       key "action", INT, value_buffer_size == num_envs
 *   observations  key "screen", BYTE, num_envs * 12288 values (env-major, 64x64x3 RGB)
 *   step infos    (num_envs > 1 only) "reward" FLOAT[num_envs], "terminated" BYTE[num_envs],
 *                 "truncated" BYTE[num_envs]; the scalar step_data fields mirror env 0;
 *                 device-resident results (also reset infos): "screen_device", "reward_device", "terminated_device",
 *                 "truncated_device", "stream" — INT[2 * num_devices], the (low, high) 32-bit halves of the CUDA device
 *                 address of each device shard's buffer (uint8 [count * 12288] / float [count] / uint8 [count]) and of
 *                 the cudaStream_t its kernels run on; the same addresses come from cenv_device_buffer(key, shard).
 *                 Host result buffers are page-locked.
 *                 With "final_observation" the step infos add "final_screen_device" (INT[2 * num_devices], as above:
 *                 uint8 [count * 12288] per shard, also cenv_device_buffer("final_screen", shard)) and, with host_copy,
 *                 "final_screen" (BYTE[num_envs * 12288]). Row i of either is written in a step iff env i terminated or
 *                 was truncated in it (the rows of the other envs keep older contents; zero at cenv_make); only those
 *                 rows are copied to the host.
 * With num_envs == 1 and no extension option the behaviour is the reference's.
 */
#ifndef PG2_CENV_H
#define PG2_CENV_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define CENV_API __declspec(dllexport)
#else
#define CENV_API __attribute__((__visibility__("default")))
#endif

#define CENV_VERSION 1

/* tags 0-3: element type of a value / buffer; tags 4-5: space descriptors */
typedef enum {
    CENV_VALUE_TYPE_INT = 0,             /* int32_t */
    CENV_VALUE_TYPE_FLOAT = 1,           /* float   */
    CENV_VALUE_TYPE_DOUBLE = 2,          /* double  */
    CENV_VALUE_TYPE_BYTE = 3,            /* uint8_t */
    CENV_SPACE_TYPE_BOX = 4,             /* float buffer: lows then highs */
    CENV_SPACE_TYPE_MULTI_DISCRETE = 5   /* int32 buffer: nvec */
} cenv_value_type;

typedef union { int32_t i; float f; double d; uint8_t b; } cenv_value;
typedef union { int32_t* i; float* f; double* d; uint8_t* b; } cenv_value_buffer;

/* named, typed buffer (observation, action, info, space) */
typedef struct {
    const char* key;
    cenv_value_type value_type;
    int32_t value_buffer_size;
    cenv_value_buffer value_buffer;
} cenv_key_value;

/* named scalar option for make / reset */
typedef struct {
    const char* name;
    cenv_value_type value_type;
    cenv_value value;
} cenv_option;

typedef struct {
    int32_t observation_spaces_size;
    cenv_key_value* observation_spaces;
    int32_t action_spaces_size;
    cenv_key_value* action_spaces;
} cenv_make_data;

typedef struct {
    int32_t observations_size;
    cenv_key_value* observations;
    int32_t infos_size;
    cenv_key_value* infos;
} cenv_reset_data;

typedef struct {
    int32_t observations_size;
    cenv_key_value* observations;
    cenv_value reward;
    bool terminated;
    bool truncated;
    int32_t infos_size;
    cenv_key_value* infos;
} cenv_step_data;

/* frame of cenv_render(): element (x, y, ch) at ch + channels * (x + width * y) */
typedef struct {
    cenv_value_type value_type;
    int32_t value_buffer_width;
    int32_t value_buffer_height;
    int32_t value_buffer_channels;
    cenv_value_buffer value_buffer;
} cenv_render_data;

/* result structs, owned by the library, read by the caller after each call */
CENV_API extern cenv_make_data make_data;
CENV_API extern cenv_reset_data reset_data;
CENV_API extern cenv_step_data step_data;
CENV_API extern cenv_render_data render_data;

/* entry points; 0 = success */
CENV_API int32_t cenv_get_env_version();
CENV_API int32_t cenv_make(const char* render_mode, cenv_option* options, int32_t options_size);
CENV_API int32_t cenv_reset(cenv_option* options, int32_t options_size);
CENV_API int32_t cenv_step(cenv_key_value* actions, int32_t actions_size);
CENV_API int32_t cenv_render();
CENV_API void cenv_close();

/* Extension (not in the reference): CUDA device address of the result buffer `key` ("screen" | "reward" | "terminated" |
 * "truncated" | "final_screen" | "stream") of device shard `device_index`; NULL if unknown / not made ("final_screen":
 * without "final_observation"). */
CENV_API void* cenv_device_buffer(const char* key, int32_t device_index);

#ifdef __cplusplus
}
#endif
#endif
