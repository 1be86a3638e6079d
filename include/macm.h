/*
 * macm.h -- C ABI of libmacm.so: the B200-native batched replacement for the one hot path of
 * siyarvurucu/gym-macm (per-step Box2D world update + reward pass + observation pass over
 * thousands of independent environments).
 *
 * The reference has no FFI layer of its own: its Python hosts (gym_macm/envs/mvmnt.py,
 * gym_macm/envs/combat.py, gym_macm/cm_framework.py) drive the pybox2d SWIG module call by
 * call.  Each entry point below names the reference interface it subsumes (file:line into the
 * reference tree).  INTEGRATION.md shows the ctypes stub a maintainer adds on the reference
 * side.
 *
 * Conventions
 *   - plain C: pointers, sizes, ints; no C++/torch types.  `stream` is a cudaStream_t passed
 *     as void* (NULL = the legacy default stream).
 *   - every pointer in macm_buffers is a DEVICE pointer owned by the caller (the Python host
 *     allocates them as torch CUDA tensors); the library only keeps the addresses.
 *   - layout: env-major, agent-minor, fp32/int32/uint8 SoA.  Agent i of env e is element
 *     e*N + i of every per-agent array.
 *   - return value: MACM_OK (0) or a negative macm_status; never throws, never exits.
 *   - no host synchronisation inside macm_step / macm_observe / macm_reset / macm_bot_actions;
 *     only the *_host convenience calls synchronise (on their own stream).
 *   - a handle is thread-compatible (one thread at a time), not thread-safe.
 *   - there is no CPU fallback: without a CUDA device macm_create fails with MACM_E_CUDA.
 */
#ifndef MACM_H
#define MACM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MACM_ABI_VERSION 8
#define MACM_MAX_AGENTS 128  /* per environment (the reference has no cap, mvmnt.py:61); up to 64: two agents per lane,
                                beyond: four, with 128-bit contact adjacency rows */
#define MACM_MAX_TARGETS 16
#define MACM_MAX_TEAMS 8

typedef enum macm_status {
    MACM_OK = 0,
    MACM_E_INVALID = -1,     /* bad argument / parameter out of range */
    MACM_E_CUDA = -2,        /* a CUDA runtime call failed; see macm_last_cuda_error */
    MACM_E_UNBOUND = -3,     /* macm_bind has not been called or a required buffer is NULL */
    MACM_E_ALIGN = -4,       /* a bound buffer is not aligned to its vector width */
    MACM_E_NOMEM = -5,
    MACM_E_UNSUPPORTED = -6  /* valid request that this build does not implement */
} macm_status;

enum { MACM_ENV_FLOCK = 0, MACM_ENV_TDM = 1 };
enum { MACM_REWARD_BINARY = 0, MACM_REWARD_LINEAR = 1 };
enum { MACM_ACTION_DISCRETE = 0, MACM_ACTION_CONTINUOUS = 1 };
enum { MACM_COORD_POLAR = 0, MACM_COORD_CARTESIAN = 1 };
/* macm_params.obs_dtype: the element type of every observation the library stores.  The values are computed in fp32
 * as always; a 16-bit type rounds each one once, to nearest even, at the store.  Nothing else changes: state,
 * rewards, nn_idx, collided, done and the trajectory are those of MACM_OBS_F32. */
enum { MACM_OBS_F32 = 0, MACM_OBS_F16 = 1, MACM_OBS_BF16 = 2 };
/* Box2D <= 2.3.0: v *= clamp(1 - h*c, 0, 1);  Box2D >= 2.3.1: v *= 1 / (1 + h*c) */
enum { MACM_DAMPING_TAYLOR = 0, MACM_DAMPING_PADE = 1 };
/* macm_params.flags */
enum {
    MACM_FLAG_REPAIR_MOV_COOLDOWN = 1, /* SURVEY App. B10: cooldown_mov_penalty counts down */
    MACM_FLAG_AUTO_RESET = 2           /* every macm_step / macm_rollout launch is followed by macm_reset_masked(NULL):
                                          envs whose `done` flag is set start a new episode (see macm_reset_masked);
                                          inside a macm_rollout launch the same reset happens after every step, so the
                                          per-step outputs are those of n_steps single steps with the flag set; the
                                          finished episode's terminal rows go to the final destinations first
                                          (macm_bind_final, macm_rollout_out.final_*) */
};
/* env_state[e][1]: bits 0-2 flags, bits 8-31 the env's episode counter (incremented by macm_reset_masked) */
enum {
    MACM_ENV_FRESH = 1,           /* world has new fixtures: FindNewContacts runs at the start of the next step */
    MACM_ENV_CONTACT_OVERFLOW = 2,/* more live contacts than max_contacts: newest were dropped (sticky until reset) */
    MACM_ENV_TOUCH_OVERFLOW = 4   /* more touching contacts than max_touching: solver skipped the excess (sticky) */
};
#define MACM_ENV_EPISODE_SHIFT 8
/* scripted actors of test_scripts/bots.py, run on the device by macm_bot_actions */
enum { MACM_BOT_IDLE = 0, MACM_BOT_FORWARD = 1, MACM_BOT_ROTATE = 2, MACM_BOT_DIAG = 3,
       MACM_BOT_FLOCK = 4, MACM_BOT_RANDOM = 5, MACM_BOT_COMBAT = 6 /* bots.py:3-16, TDM only */,
       MACM_BOT_CIRCLE = 7 /* bots.py:31-35 */ };

/*
 * Everything gym_macm/settings.py and the Agent classes hold that the hot path reads.
 * Doubles stay doubles because the reference's host arithmetic is Python float64
 * (mvmnt.py:103-116); the library rounds to fp32 exactly where pybox2d's SWIG layer does.
 */
typedef struct macm_params {
    int32_t env_kind;             /* MACM_ENV_* : Flock (mvmnt.py:27) or TDM (combat.py:56) */
    int32_t n_envs;               /* independent worlds in the batch */
    int32_t n_agents;             /* sum(n_agents) of the ctor (mvmnt.py:61), 2..MACM_MAX_AGENTS */
    int32_t n_targets;            /* len(unique(targets)) (mvmnt.py:42), 1..MACM_MAX_TARGETS; TDM: 0 */
    int32_t max_contacts;         /* contact capacity per env; 0 = min(N(N-1)/2, 8N) */
    int32_t max_touching;         /* touching-contact capacity per env; 0 = min(max_contacts, 2N) up to 64 agents, and beyond 64 a
                                     shared stage of min(2N, 192) with a global-memory one of min(max_contacts, 3N) behind
                                     it (a flock gathered at its target reaches ~1.8N).  Up to 240 the solver's stage lives
                                     in shared memory; a larger value adds a global-memory stage (macm_buffers.touch_scratch,
                                     32 bytes per contact and env) that takes the env with more touching contacts than the
                                     shared stage holds -- exact, slow, for gathered flocks and dense spawn piles.
                                     macm_buffer_sizes.max_touching reports the effective capacity */
    double hz;                    /* settings.py:30   60.0 */
    int32_t velocity_iterations;  /* settings.py:31   8 */
    int32_t position_iterations;  /* settings.py:32   3 */
    int32_t warm_starting;        /* settings.py:34   1 */
    int32_t damping_model;        /* MACM_DAMPING_*   (pybox2d's engine version is unpinned; default PADE: pip releases bundle Box2D >= 2.3.1) */
    double radius;                /* settings.py:128  0.5 */
    double density;               /* settings.py:130  1 */
    double friction;              /* settings.py:131  0.3 */
    double linear_damping;        /* settings.py:133  5 */
    double agent_force;           /* settings.py:124  20 */
    double agent_rotation_speed;  /* settings.py:123  0.8 * 2 pi */
    double time_limit;            /* settings.py:125  60 */
    int32_t reward_mode;          /* settings.py:137 */
    int32_t action_mode;          /* settings.py:136 */
    int32_t coord;                /* settings.py:141 */
    int32_t flags;                /* MACM_FLAG_* */
    double reward_radius;         /* settings.py:146  7 (binary) */
    /* TDM only: combat.py:20-24, settings.py:165-166 */
    double cooldown_atk;          /* 1 */
    double cooldown_mov_penalty;  /* 0.5 */
    double melee_range;           /* 2 */
    double melee_dmg;             /* 0.25 */
    double percent_mov_penalty;   /* 0.2 */
    double init_health;           /* 1 */
    /* initial-state distributions, used only by macm_sample_reset */
    double start_spread;          /* settings.py:121  20   Flock: pos = spread * (U - 0.5) + start_point */
    double start_x, start_y;      /* settings.py:122  0, 0 */
    double target_mindist;        /* settings.py:139  25 */
    double target_maxdist;        /* settings.py:140  60 */
    double world_width;           /* combat.py:76     30   TDM: x = U * (team + width/2), y = U * height */
    double world_height;          /* combat.py:77     30 */
    int32_t env_index_base;       /* global index of env 0 of this handle (shards of one batch); keys the samplers */
    int32_t obs_dtype;            /* MACM_OBS_*: element type of `obs` and of every other observation destination */
} macm_params;

/* Caller-owned device buffers.  E = n_envs, N = n_agents, T = n_targets, C = max_contacts. */
typedef struct macm_buffers {
    /* ---- state (read and written by macm_step) ---- */
    float* posvel;            /* [E,N,4] x y vx vy                      16-byte aligned */
    float* angsleep;          /* [E,N,2] body angle, b2Body::m_sleepTime  8-byte aligned */
    float* fat;               /* [E,N,4] broadphase fat AABB lo.x lo.y hi.x hi.y  16-byte aligned */
    uint32_t* contact_ab;     /* [E,C]   a | b<<8 | touching<<16, in BIRTH order (oldest first), a < b */
    float* contact_imp;       /* [E,C,2] normalImpulse, tangentImpulse (warm start)  8-byte aligned */
    int32_t* contact_count;   /* [E] */
    int32_t* env_state;       /* [E,4]   step_count, MACM_ENV_* bits, touching contacts of the last step, winner (TDM; -1)  16-byte aligned */
    float* targets;           /* [E,T,2] Flock target positions (mvmnt.py:47-52)  8-byte aligned */
    uint8_t* target_idx;      /* [N]     targets_idx (mvmnt.py:43), shared by all envs */
    float* tdm_state;         /* [E,N,4] TDM: health, cooldown_atk steps left (int bits), cooldown_mov steps left (int bits), alive | hits_taken<<8 (int bits)  16-byte aligned */
    uint8_t* team;            /* [N]     TDM: team of agent i, shared by all envs */
    /* ---- outputs (written by macm_step / macm_observe) ---- */
    float* obs;               /* Flock polar [E,N,4] = nn_dist nn_theta tgt_r tgt_theta;
                                 Flock cartesian [E,N,6] = nn_dist nn_cos nn_sin tgt_r tgt_cos tgt_sin;
                                 TDM [E,N,N,4] = r theta phi type(1 ally, 0 enemy, -1 no entry)   16-byte aligned.
                                 With a 16-bit obs_dtype the member points at fp16 / bf16 elements of the same layout,
                                 and the alignment is that of one record: 8 bytes (Flock polar, TDM) or 4 bytes (Flock
                                 cartesian, 12-byte records).  The same holds for every other `obs` pointer below */
    int32_t* nn_idx;          /* [E,N] id of the nearest other agent (mvmnt.py:187-196); TDM: unused */
    float* rewards;           /* [E,N] */
    uint8_t* collided;        /* [E,N] agent appears in some world contact (mvmnt.py:162-164) */
    uint8_t* done;            /* [E] */
    /* ---- scratch (max_touching > 240, or the default beyond 64 agents; see macm_buffer_sizes.touch_scratch) ---- */
    uint8_t* touch_scratch;   /* the solver's stage of an env with more touching contacts than shared memory holds  16-byte aligned */
} macm_buffers;

/* Bytes each macm_buffers member must hold for this sim (0 = not used by this env kind). */
typedef struct macm_buffer_sizes {
    uint64_t posvel, angsleep, fat, contact_ab, contact_imp, contact_count, env_state, targets,
             target_idx, tdm_state, team, obs, nn_idx, rewards, collided, done, touch_scratch;
    int32_t obs_dim;          /* values per agent in `obs` (`obs` bytes = E * N * obs_dim * element size of obs_dtype) */
    int32_t action_bytes;     /* bytes per agent in the `actions` argument of macm_step */
    int32_t max_contacts, max_touching;
} macm_buffer_sizes;

/* Launch geometry and derived constants, for benchmarks / DESIGN.md. */
typedef struct macm_launch_info {
    int32_t lanes_per_env, agents_per_lane, envs_per_block, threads_per_block, blocks;
    int32_t smem_bytes_per_block, blocks_per_sm, sm_count;
    int32_t done_step;        /* first step on which done becomes true (3601 for the defaults, mvmnt.py:134-136) */
    float dt, dt_ratio, inv_mass, damping_factor, binary_d2_threshold;
} macm_launch_info;

typedef struct macm_sim macm_sim;

int macm_abi_version(void);
const char* macm_strerror(int status);
/* Text of the last CUDA error seen by this handle ("" if none). */
const char* macm_last_cuda_error(const macm_sim* sim);

/* Fill *p with the reference defaults: flockSettings (settings.py:110-146) or combatSettings
 * (settings.py:149-175) + combat.Agent constants (combat.py:20-24) + fwSettings (settings.py:25-36). */
int macm_params_default(macm_params* p, int env_kind);

/* Replaces world construction: NoRender(settings) -> FrameworkBase.__init__ ->
 * b2World(gravity=(0,0), doSleep=True) (cm_framework.py:155-167) for n_envs worlds at once.
 * Validates the parameters, derives the fp32 engine constants, selects device `device`.
 * No device memory is allocated here except two small tables and, lazily, the staging of the *_host calls.
 * On MACM_E_CUDA after the device was found, *out still receives a handle whose only use is
 * macm_last_cuda_error(*out) followed by macm_destroy(*out) (which frees whatever was allocated); on every other
 * failure *out is NULL. */
int macm_create(macm_sim** out, const macm_params* p, int device);
int macm_destroy(macm_sim* sim);

int macm_get_buffer_sizes(const macm_sim* sim, macm_buffer_sizes* out);
int macm_get_launch_info(const macm_sim* sim, macm_launch_info* out);
int macm_bind(macm_sim* sim, const macm_buffers* buffers);

/* Replaces body creation, world.CreateDynamicBody(**bodySettings, position, angle) for every
 * agent (mvmnt.py:61-76, combat.py:82-98) plus `self.obs = self.get_obs()` (mvmnt.py:79):
 * reads posvel (x, y, vx, vy), angsleep.angle, targets; writes fat = tight AABB +- 0.1
 * (b2_aabbExtension), sleep time 0, no contacts, step_count 0, MACM_ENV_FRESH; TDM: health =
 * init_health, cool-downs 0, alive 1; then the observation pass. */
int macm_reset(macm_sim* sim, void* stream);

/* Samples initial states on the device with the reference's distributions (mvmnt.py:48-52,
 * 62-64; combat.py:84-86) from a counter-based generator keyed by (seed, env, agent), then
 * does what macm_reset does.  The reference draws from Python's unseeded `random`. */
int macm_sample_reset(macm_sim* sim, uint64_t seed, void* stream);

/* Per-env reset: a new episode for some envs of the batch, the others untouched -- the reference's `env.reset()`
 * (mvmnt.py:224-233, combat.py:229-239; broken as shipped, SURVEY App. B3) applied to the envs a learner has
 * seen finish (`done`: time limit mvmnt.py:134-136, one team left combat.py:171-182).
 *   mask   device uint8 [E] (non-zero = reset this env), or NULL = the bound `done` buffer.
 * A selected env gets fresh agent states and targets drawn from the reference's distributions (the draws of
 * macm_sample_reset keyed by (seed, global env, agent, episode), episode = the env's reset count, so two
 * episodes of one env differ and a batch is the same however it is sharded), then what macm_reset does for it:
 * fat AABBs, no contacts, step_count 0, MACM_ENV_FRESH, cleared overflow bits, TDM health / cool-downs /
 * alive, the first observation of the new episode in `obs` / `nn_idx`.  `rewards`, `collided` and `done` keep the
 * values of the env's last step (the learner reads the terminal reward next to the new episode's first observation;
 * the next step overwrites them).  One launch, no host synchronisation. */
int macm_reset_masked(macm_sim* sim, const uint8_t* mask, uint64_t seed, void* stream);
/* Final destinations: whenever the library resets an env -- macm_reset_masked, the launch MACM_FLAG_AUTO_RESET appends to
 * a step or rollout, a rollout's in-launch reset -- it first copies that env's rows of obs, nn_idx (Flock), tdm_state
 * (TDM) and env_state, as they stand at that moment, to the bound final arrays: the finished episode's terminal
 * observation (a time-limit end is a truncation: a learner bootstraps from it) and its outcome (step count, overflow
 * bits, TDM winner; TDM health / alive).  Rows of envs that are not reset are left untouched.  Any member may be NULL. */
typedef struct macm_final_out {
    float* obs;        /* [E,N,obs_dim]  obs_dtype elements, aligned as macm_buffers.obs (16 bytes in fp32) */
    int32_t* nn_idx;   /* [E,N]          Flock only */
    float* tdm_state;  /* [E,N,4]        TDM only, 16-byte aligned */
    int32_t* env_state;/* [E,4]          16-byte aligned */
} macm_final_out;
/* Binds (the addresses are kept; caller-owned device memory) or, with f == NULL, unbinds the final arrays.
 * MACM_E_ALIGN: a misaligned member; MACM_E_INVALID: nn_idx on TDM or tdm_state on Flock.  Nothing bound: no copies. */
int macm_bind_final(macm_sim* sim, const macm_final_out* f);
/* Seed of the resets that MACM_FLAG_AUTO_RESET appends to every step (default 0). */
int macm_set_auto_reset_seed(macm_sim* sim, uint64_t seed);
/* Device-side overflow summary: *contact_envs / *touching_envs receive how many envs currently carry
 * MACM_ENV_CONTACT_OVERFLOW / MACM_ENV_TOUCH_OVERFLOW (results of such an env differ from the reference's from
 * the overflowing step on).  Synchronises `stream`.  Either pointer may be NULL. */
int macm_overflow_count(macm_sim* sim, int32_t* contact_envs, int32_t* touching_envs, void* stream);

/* Replaces one Flock.step / TDM.step for every env (mvmnt.py:81-140, combat.py:104-184):
 * action decode -> ApplyForce, framework.Step -> b2World::Step(1/hz, velIters, posIters) +
 * ClearForces (cm_framework.py:213-224), get_rewards (mvmnt.py:160-179), time/done
 * (mvmnt.py:134-136), get_obs (mvmnt.py:181-222 / combat.py:206-227).
 * actions (device): discrete uint8 [E,N,4] = a0 a1 a2 a3 (a3: TDM attack bit; Flock ignores it),
 *                   continuous float [E,N,2]. */
int macm_step(macm_sim* sim, const void* actions, void* stream);

/* Per-step outputs of macm_rollout: caller-owned device arrays with a leading step axis; any member may be NULL. */
typedef struct macm_rollout_out {
    float* obs;        /* [K,E,N,obs_dim]  obs_dtype elements, aligned as macm_buffers.obs (16 bytes in fp32) */
    int32_t* nn_idx;   /* [K,E,N]          (Flock) */
    float* rewards;    /* [K,E,N] */
    uint8_t* collided; /* [K,E,N] */
    uint8_t* done;     /* [K,E] */
    /* Terminal rows of the envs reset after step k (MACM_FLAG_AUTO_RESET on and done[k][e] set), as macm_bind_final
     * describes; row [k][e] is written iff env e was reset after step k, every other row is left untouched. */
    float* final_obs;        /* [K,E,N,obs_dim]  obs_dtype elements, aligned as macm_buffers.obs (16 bytes in fp32) */
    int32_t* final_nn_idx;   /* [K,E,N]          Flock only */
    float* final_tdm_state;  /* [K,E,N,4]        TDM only, 16-byte aligned */
    int32_t* final_env_state;/* [K,E,4]          16-byte aligned */
} macm_rollout_out;

/* n_steps consecutive Flock.step / TDM.step calls for every env in ONE launch -- the reference's
 * `for _ in range(n_steps): obs, rewards = env.step(actions_k)` loop (README.md:8-14).  Every env runs its
 * n_steps steps back to back with its bodies, fat AABBs and clocks held on chip; only the actions (in), the
 * per-step outputs (out) and the contact lists touch HBM between the steps.  Bit-identical to n_steps calls
 * of macm_step: the bound state and output buffers end up exactly as after the last of those calls, and
 * out->x[k] holds what buffer x held after call k.  The same holds for the bound final arrays (each holds the latest
 * terminal row of its env) and out->final_x[k] holds what final array x received from the reset after call k.
 *   actions != NULL : [n_steps,E,N,4] uint8 (discrete) or [n_steps,E,N,2] float (continuous), device.
 *   actions == NULL : the actions=None mode (mvmnt.py:86-92): every agent's actor picks its action from
 *                     its own last observation, policy = MACM_BOT_* as in macm_bot_actions (MACM_BOT_FLOCK: Flock
 *                     with polar coordinates; MACM_BOT_COMBAT: TDM), draws keyed by (seed, env, agent, step_count).
 * With out == NULL or out->obs == NULL the observation pass only runs after the last step (action repeat /
 * frame skip); rewards of the intermediate steps are still available through out->rewards.
 * With a 16-bit obs_dtype, policy MACM_BOT_FLOCK returns MACM_E_UNSUPPORTED: its first step would steer by the rounded
 * stored observation and so leave the fp32 trajectory.  MACM_BOT_COMBAT recomputes its row in fp32 and stays. */
int macm_rollout(macm_sim* sim, const void* actions, int32_t n_steps, int32_t policy, uint64_t seed,
                 const macm_rollout_out* out, void* stream);

/* get_obs() alone on the current state (mvmnt.py:181-222 / combat.py:206-227). */
int macm_observe(macm_sim* sim, void* stream);

/* test_scripts/bots.py on the device: writes one action per agent from the current `obs`
 * buffer (`actions=None` mode, mvmnt.py:86-92).  MACM_BOT_RANDOM draws U{0,1,2}^3 (x U{0,1}) and
 * MACM_BOT_CIRCLE its coin keyed by (seed, env, agent, step_count); MACM_BOT_COMBAT (TDM) faces, approaches and
 * strikes the nearest enemy of the agent's observation row (bots.py:3-16).
 * MACM_BOT_FLOCK and MACM_BOT_COMBAT read the stored `obs`; with a 16-bit obs_dtype they return MACM_E_UNSUPPORTED
 * (a rounded observation would change their decisions).  The other policies do not read it and stay supported. */
int macm_bot_actions(macm_sim* sim, int policy, uint64_t seed, void* actions_out, void* stream);

/* Any little-endian integer array [E,N,width] (width 3 = a0 a1 a2, or 4 = + attack; elements of 1, 2, 4 or 8
 * bytes, device memory) -> the uint8 [E,N,4] action words macm_step reads (actions dict -> array, mvmnt.py:94-101). */
int macm_pack_actions(macm_sim* sim, const void* src, int32_t elem_bytes, int32_t width, void* actions_out, void* stream);

/* The drop-in boundary with HOST buffers: copies `actions` host->device, steps, copies
 * obs / rewards / nn_idx / collided / done device->host (any of the outputs may be NULL) and
 * waits.  Pinned host memory (macm_host_alloc) makes the copies asynchronous DMA.  Outputs that lie back to
 * back in device memory AND in host memory (same offsets, gaps under 256 bytes) travel in ONE transfer.
 * The handle's stream is ordered after everything the other entry points enqueued for this handle before the
 * call, and their later launches after it (events recorded at the hand-over, none between two steps). */
int macm_step_host(macm_sim* sim, const void* actions, float* obs, float* rewards, int32_t* nn_idx,
                   uint8_t* collided, uint8_t* done);
/* The same work enqueued on the handle's own stream without waiting: with pinned host buffers the
 * copies and the kernel of one batch overlap those of another batch (two handles in ping-pong).
 * The outputs are valid after macm_host_sync(sim).  The host state (bound device buffers) of a
 * handle must not be touched from other streams between the two calls. */
int macm_step_host_async(macm_sim* sim, const void* actions, float* obs, float* rewards, int32_t* nn_idx,
                         uint8_t* collided, uint8_t* done);
int macm_host_sync(macm_sim* sim);
int macm_host_alloc(void** out, uint64_t bytes);
int macm_host_free(void* p);

/* Lets kernels running on `device` load and store memory that lives on `peer_device` (NVLink / PCIe peer access;
 * idempotent).  Needed once per process before a macm_rollout_out pointer may name another GPU's buffer -- the
 * learner-side gather of BASELINE config 5 done by the step kernel itself (gym_macm.dist.PeerGather). */
int macm_enable_peer_access(int device, int peer_device);
/* A zeroed device allocation of its own (cudaMalloc, not a slice of the host framework's pool) together with the
 * 64 bytes of its cudaIpcMemHandle_t (ipc_handle_out may be NULL): what the learner rank exports to the others. */
int macm_device_alloc(int device, uint64_t bytes, void** out, void* ipc_handle_out);
int macm_device_free(void* p);
/* Maps a device allocation exported by another process of the box (`handle` = the 64 bytes of its
 * cudaIpcMemHandle_t) for kernels running on `device`; *out receives the base address of the allocation. */
int macm_ipc_open(const void* handle, int device, void** out);
int macm_ipc_close(void* base);

/* Top-down RGB frames of some envs of the batch: what the reference's renderer shows (bodies as solid circles with their
 * heading axis, targets as white circles; see gym_macm/render.py), drawn on the device from the bound state.
 * Frame b draws env e = envs[b] with view (cx, cy, hw) = views[b]: s = W / (2 hw) pixels per metre, a world point
 * (x, y) lands on u = (x - cx) s + W/2, v = (cy - y) s + H/2 (world +y up, row 0 at the top), and pixel (row i,
 * column j) is sampled at its centre (j + 0.5, i + 0.5).  The background is black; a pixel takes the colour of the last
 * primitive that covers it, in this order:
 *   every agent i = 0..N-1, centre c, radius rho = radius s, colour col = palette[i][alt] (alt: Flock `collided`,
 *   TDM dead): the disc |p - c|^2 <= rho^2 in col >> 1 per channel, the outline (rho - 1)^2 < |p - c|^2 <= rho^2 in
 *   col (rho < 1: the whole disc), then the heading axis, the pixels within 0.5 px of the segment from c to
 *   c + rho (cos angle, -sin angle), in col;
 *   Flock: every target t = 0..T-1 as an outline ring of radius reward_radius s in white.
 * A frame whose env index lies outside [0, n_envs), or whose half-width is not a finite value > 0, is left black
 * (envs and views are device data: the call does not read them on the host).  Reads the bound state, writes only
 * `out`; one launch, no host synchronisation.  MACM_E_INVALID: a size out of range, a NULL views / palette / out, or
 * envs == NULL with n_frames > n_envs; MACM_E_ALIGN: views or envs not 4-byte aligned; MACM_E_UNBOUND: before
 * macm_bind. */
typedef struct macm_render_args {
    int32_t n_frames;        /* B >= 1 */
    int32_t height, width;   /* H, W in 1..4096 */
    const int32_t* envs;     /* [B] device: the env drawn in frame b; NULL = frame b draws env b (B <= n_envs) */
    const float* views;      /* [B,3] device: centre x, centre y, half-width in metres of frame b (half-width > 0) */
    const uint8_t* palette;  /* [N,2,3] device: per agent, the RGB bytes of its normal and of its alternate colour */
    uint8_t* out;            /* [B,H,W,3] device, row 0 at the top */
} macm_render_args;
int macm_render(macm_sim* sim, const macm_render_args* a, void* stream);

/* Agent-centred RGB frames: every agent's own view of its env, heading up, drawn on the device from the bound state
 * (what a decentralised pixel policy sees).  Frame (b, i) looks at env e = envs[b] from agent i: its centre (cx, cy)
 * is the agent's fp32 position, its heading ci = cos a_i, si = sin a_i (float64, of the fp32 body angle), and
 * s = W / (2 half_width) pixels per metre.  A world point (x, y), dx = x - cx, dy = y - cy, lands on
 *   u = W/2 + s (dx si - dy ci),   v = H/2 - s (dx ci + dy si),
 * so the agent's heading points to the top of the frame and its right-hand side is on the right.  The heading axis
 * of agent k (ck, sk) runs along the pixel direction (ck si - sk ci, -(ck ci + sk si)): agent i's own points straight
 * up.  Everything else is macm_render's rules: pixel centres at (j + 0.5, r + 0.5); agents as discs at half the
 * colour with an outline and a heading axis within 0.5 px, of radius rho = radius s and axis length rho; Flock
 * targets as white rings of radius reward_radius s; palette[i][1] for a Flock agent in a contact or a dead TDM agent;
 * a black background; the last primitive in painter's order (agents 0..N-1, then targets 0..T-1) wins.  A dead TDM
 * agent still gets its frame: its body stays in the world.
 * An env index outside [0, n_envs) gives N black frames and reads no state for that row (envs is device data: the
 * call does not read it on the host).  Reads the bound state, writes only `out`; one launch, no host synchronisation.
 * MACM_E_INVALID: a size out of range, a half_width that is not finite and > 0, a NULL palette / out, or envs == NULL
 * with B > n_envs; MACM_E_ALIGN: envs not 4-byte aligned; MACM_E_UNBOUND: before macm_bind. */
typedef struct macm_agent_frames_args {
    int32_t n_envs;          /* B >= 1 envs; every agent of each gets a frame */
    int32_t height, width;   /* H, W in 1..1024 */
    double half_width;       /* metres from the frame centre to its left / right edge; finite, > 0 */
    const int32_t* envs;     /* [B] device: env of frame row b; NULL = env b (B <= n_envs of the sim) */
    const uint8_t* palette;  /* [N,2,3] device, as macm_render */
    uint8_t* out;            /* [B,N,H,W,3] device: frame (b, i) is agent i of env envs[b], row 0 at the top */
} macm_agent_frames_args;
int macm_render_agents(macm_sim* sim, const macm_agent_frames_args* a, void* stream);

/* Lidar scans: every agent's fan of R closest-hit ray casts around its heading, cast on the device from the bound
 * state (the range sensor of swarm policies).  Row b scans env e = envs[b] (env b when envs is NULL).  For agent i of
 * that env and ray r = 0..R-1:
 *   origin     p1 = the agent's fp32 centre (x, y);
 *   direction  float64, in this order: o_r = fov * ((double)(2r + 1 - R) / (double)(2R)), th = (double)a_i + o_r
 *              (a_i the fp32 body angle), dx = (float)(L * cos(th)), dy = (float)(L * sin(th)), L = max_range;
 *   end        p2 = (x + dx, y + dy), added in fp32 (the TDM attack's ray, with L for melee_range).
 * The fan is symmetric about the heading (cos a_i, sin a_i); r counts counter-clockwise, and with an odd R the middle
 * ray points straight ahead.  The hit is the closest-hit cast of the step's TDM attack (cm_framework.py:56-86):
 * b2CircleShape::RayCast in fp32 and Box2D's operation order, with the fp32 radius and maxFraction 1, against every
 * body that has a proxy -- a dead TDM agent has none, so rays pass through it (a dead agent still scans: its body
 * stays in the world).  The smallest fraction wins; among equal fractions, the lowest agent index.  Nothing special-
 * cases the caster: a ray whose origin lies inside a disc (in the fp32 arithmetic, |p1 - c|^2 < radius^2) gets
 * a = -(c + sqrt(sigma)) <= 0 from it, so the disc is never reported at a fraction above 0.  The caster's own disc
 * (p1 - c = 0, a < 0) is never reported at all; a neighbour's disc holding the origin is reported only at fraction
 * +-0, when the origin sits on its rim to within rounding.
 * Output: fraction[b][i][r] in [0, 1], 1 = no hit, computed in fp32 and rounded once, to nearest even, to the sim's
 * obs_dtype at the store (it is an observation); hit[b][i][r] = the agent id hit, or -1 (int32, like nn_idx).
 * An env index outside [0, n_envs) gives a row of misses (fraction 1, hit -1) and reads no state for that row (envs
 * is device data: the call does not read it on the host).  Reads the bound state, writes only its outputs; one
 * launch, no host synchronisation.
 * MACM_E_INVALID: an argument out of range, a NULL fraction, or envs == NULL with B > n_envs; MACM_E_ALIGN: envs or
 * hit not 4-byte aligned, or fraction not aligned to its element; MACM_E_UNBOUND: before macm_bind. */
#define MACM_MAX_RAYS 1024
typedef struct macm_lidar_args {
    int32_t n_envs;          /* B >= 1 env rows; every agent of each gets a scan */
    int32_t n_rays;          /* R in 1..MACM_MAX_RAYS */
    double max_range;        /* L, metres: finite, > 0, <= 1e6 */
    double fov;              /* radians: finite, 0 < fov <= 2 pi */
    const int32_t* envs;     /* [B] device, or NULL = env b (B <= n_envs of the sim) */
    void* fraction;          /* [B,N,R] obs_dtype elements */
    int32_t* hit;            /* [B,N,R] device, or NULL */
} macm_lidar_args;
int macm_lidar(macm_sim* sim, const macm_lidar_args* a, void* stream);

/* Number of kernels this handle has launched so far. */
int64_t macm_launch_count(const macm_sim* sim);

/* Profiling hook (no reference counterpart): when `trace` is a device buffer of n_envs x 4 uint64,
 * every step launch records per env {%globaltimer at entry (ns), %globaltimer at exit (ns), SM cycles
 * spent, smid | touching<<16 | islands<<32 | multi<<48 | slot<<49}.  NULL switches it off (the default). */
int macm_set_trace(macm_sim* sim, void* trace);

#ifdef __cplusplus
}
#endif
#endif /* MACM_H */
