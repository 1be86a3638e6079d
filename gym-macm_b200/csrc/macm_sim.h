// Internal definitions shared by the kernels (macm_kernels.cu) and the C-ABI (macm_api.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "macm.h"

// b2Settings.h of Box2D 2.3.0 -- the engine pybox2d wraps (SURVEY.md Appendix A.1).
#define B2_PI 3.14159265359f
#define B2_EPSILON 1.192092896e-07f
#define B2_AABB_EXTENSION 0.1f
#define B2_AABB_MULTIPLIER 2.0f
#define B2_LINEAR_SLOP 0.005f
#define B2_MAX_LINEAR_CORRECTION 0.2f
#define B2_MAX_TRANSLATION 2.0f
#define B2_BAUMGARTE 0.2f
#define B2_TIME_TO_SLEEP 0.5f
#define B2_LINEAR_SLEEP_TOLERANCE 0.01f
// numpy's float64 pi (mvmnt.py:105-106,114,199)
#define NP_PI 3.141592653589793

// Kernel argument block (passed by value as a __grid_constant__).
struct SimConst {
    int E, N, T, C, TC;
    int kind, reward_mode, action_mode, coord, vel_iters, pos_iters, warm_starting, flags;
    int done_step, cd_atk_steps, cd_mov_steps, obs_dim;
    int env_base;       // global index of this handle's env 0 (keys the counter-based samplers)
    float h;            // (float)(1/hz): timeStep at the SWIG boundary (cm_framework.py:182,222)
    float dt_ratio;     // fl(fl(1/h) * h): b2TimeStep::dtRatio once inv_dt0 != 0
    float inv_mass;     // 1 / (density * b2_pi * r * r)
    float friction;     // b2MixFriction = sqrtf(f * f)
    float damp;         // per-step linear damping factor
    float radius, rsum2;
    float k_sum, normal_mass;
    float binary_thr;   // fp32 d^2 threshold equivalent to sqrt64(d2) < reward_radius (mvmnt.py:177)
    float melee_dmg, init_health;
    int obs_dtype;      // MACM_OBS_*: element type of every observation store
    int obs_words;      // 32-bit words per agent of an observation row: obs_dim (fp32) or obs_dim / 2 (16-bit)
    double rot_step;   // agent_rotation_speed * (1/hz)       (mvmnt.py:103-104)
    double force;       // agent_force                           (mvmnt.py:113-116)
    double force_pen;   // agent_force * (1 - percent_mov_penalty) (combat.py:46-49)
    double diag;        // 1/np.sqrt(2)                          (mvmnt.py:112)
    double melee_range; // combat.py:22,145
    double melee_dmg_d; // combat.py:23,153 (health arithmetic is float64 in the reference)
    const double2* sincos_tab;  // [418] sin,cos(k/128): library-owned, filled at macm_create
    // state
    float4* posvel; float2* angsleep; float4* fat;
    uint32_t* c_ab; float2* c_imp; int* c_cnt; int4* env_state;
    const float2* targets; const uint8_t* target_idx;
    float4* tdm; const uint8_t* team;
    // outputs
    float* obs; int* nn_idx; float* rewards; uint8_t* collided; uint8_t* done;
    unsigned long long* trace;  // [E,4] per-env timing record (macm_set_trace), or null
    unsigned char* scratch;     // [E, TCH, 32] global-memory solver stage for envs with more than TC touching contacts, or null
    int TCH;                    // its capacity per env (touching contacts)
    // blocks of the step kernel that are resident at once (SMs x blocks per SM): only those can overlap their L2
    // prefetch with the predecessor's tail; a block of a later wave starts when its loads can be issued anyway
    int first_wave;
};

// Initial-state distributions (mvmnt.py:48-52,62-64; combat.py:84-86) and the key of the counter-based draws.
struct SampleConst {
    unsigned long long seed;
    double spread, sx, sy, tmin, tmax, width, height;
};

// Where a reset copies an env's rows of obs / nn_idx / tdm_state / env_state before it overwrites them: the terminal
// observation and state of the finished episode (macm_bind_final, macm_rollout_out.final_*).  Each array has the
// layout of the bound buffer of the same name; any pointer may be null.
struct Finals {
    float* obs; int* nn_idx; float4* tdm; int4* es;
};

// Arguments of a multi-step launch (macm_rollout): K consecutive steps of every env inside one kernel, the env's
// state staying on chip between them.  Per-step outputs go to the caller's [K, ...] arrays (any of them may be
// null); the sim's bound output buffers receive the last step's values, exactly as after K calls of macm_step.
// (Members are only ever appended: the single-step kernels read the leading ones at fixed parameter offsets.)
struct Rollout {
    SampleConst sc;     // distributions and seed of the in-launch resets (MACM_FLAG_AUTO_RESET)
    int K;              // steps in this launch (macm_step: 1)
    int sync;           // the block's warps start every `sync`-th step together (0 = never; 1 with one block per SM)
    int policy;         // MACM_BOT_* when `actions` is null (the actions=None mode of mvmnt.py:86-92), else -1
    unsigned long long seed;
    float* obs; int* nn_idx; float* rewards; uint8_t* collided; uint8_t* done;
    // terminal rows of the envs an in-launch reset restarts after step k < K - 1 (the reset the launch appends
    // covers step K - 1): the bound final slots [E, ...] and the caller's per-step final arrays [K, E, ...]
    Finals fin, fin_k;
    int finals;         // some pointer of fin / fin_k is set
};

struct LaunchCfg {
    int G, APL, envs_per_block, threads, blocks, smem_bytes;   // the step kernel
    int per_env_bytes;                                          // shared memory of one env
    int obs_blocks, obs_smem_bytes;                             // get_obs alone: always 128-thread blocks
};

#ifdef __CUDACC__
// Philox4x32-10 (Salmon et al., SC'11): counter-based, so a draw is a pure function of
// (seed, index, stream) and does not depend on launch geometry.
struct Philox {
    uint32_t c[4];
    __device__ Philox(uint64_t seed, uint64_t index, uint32_t stream, uint32_t sub)
    {
        uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
        c[0] = (uint32_t)index; c[1] = (uint32_t)(index >> 32); c[2] = stream; c[3] = sub;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
            const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
            c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
            k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
        }
    }
    // 53-bit uniform in [0, 1), the construction CPython's random.random() uses
    __device__ double u53(int pair) const
    {
        const uint32_t a = c[pair * 2] >> 5, b = c[pair * 2 + 1] >> 6;
        return ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);
    }
};

// One agent's initial state (mvmnt.py:62-64 / combat.py:84-86) and one target (mvmnt.py:48-52): pure functions of
// (seed, GLOBAL agent / target index, episode) -- the same draws whatever kernel or launch shape asks for them.
__device__ __forceinline__ void sample_agent(const SimConst& P, const SampleConst& sc, uint64_t gidx, int i,
                                             uint32_t episode, float& x, float& y, float& a)
{
    const Philox r(sc.seed, gidx, 0u, 2u * episode);
    const Philox r2(sc.seed, gidx, 0u, 2u * episode + 1u);
    double dx, dy;
    if (P.kind == MACM_ENV_FLOCK) {
        dx = sc.spread * (r.u53(0) - 0.5) + sc.sx;   // mvmnt.py:62-63
        dy = sc.spread * (r.u53(1) - 0.5) + sc.sy;
    } else {
        dx = r.u53(0) * ((double)P.team[i] + sc.width / 2);  // combat.py:84-85
        dy = r.u53(1) * sc.height;
    }
    x = (float)dx; y = (float)dy;
    a = (float)((-1.0 + 2.0 * r2.u53(0)) * NP_PI);   // random.uniform(-1, 1) * np.pi
}
__device__ __forceinline__ float2 sample_target(const SampleConst& sc, uint64_t gtidx, uint32_t episode)
{
    const Philox r(sc.seed, gtidx, 1u, 2u * episode);
    const double ang = 2 * NP_PI * r.u53(0);              // mvmnt.py:50-52
    const double dist = sc.tmin + r.u53(1) * (sc.tmax - sc.tmin);
    return make_float2((float)(dist * cos(ang)), (float)(dist * sin(ang)));
}
#endif

// implemented in macm_kernels.cu
cudaError_t macm_launch_cfg(const SimConst& P, int sm_count, LaunchCfg* cfg);
cudaError_t macm_prepare_kernels(const SimConst& P, const LaunchCfg& cfg, int* blocks_per_sm);
cudaError_t macm_launch_step(const SimConst& P, const LaunchCfg& cfg, const void* actions, const Rollout& R, cudaStream_t s);
cudaError_t macm_launch_observe(const SimConst& P, const LaunchCfg& cfg, cudaStream_t s);
// implemented in macm_kernels_huge.cu (the kernels with the global-memory touching stage, SimConst::scratch != null)
cudaError_t macm_prepare_kernels_huge(const SimConst& P, const LaunchCfg& cfg);
cudaError_t macm_launch_step_huge(const SimConst& P, const LaunchCfg& cfg, const void* actions, const Rollout& R, cudaStream_t s);
cudaError_t macm_launch_reset(const SimConst& P, cudaStream_t s);
// fin / fin2: where each reset env's rows go first (bound final slots; row K-1 of a rollout's final_* arrays)
cudaError_t macm_launch_reset_masked(const SimConst& P, const LaunchCfg& cfg, const uint8_t* mask, const SampleConst& sc,
                                     const Finals& fin, const Finals& fin2, cudaStream_t s);
cudaError_t macm_launch_sample(const SimConst& P, const SampleConst& sc, cudaStream_t s);
cudaError_t macm_launch_overflow_count(const SimConst& P, int* d_out2, cudaStream_t s);
cudaError_t macm_launch_pack_actions(const void* src, int elem_bytes, int width, uint64_t n_agents, void* out, cudaStream_t s);
cudaError_t macm_launch_bot(const SimConst& P, int policy, uint64_t seed, void* actions_out, cudaStream_t s);
