// macm_api.cu -- the C ABI of libmacm.so (include/macm.h): parameter validation, derivation of the
// fp32 engine constants exactly as pybox2d's SWIG boundary would round them, buffer binding,
// kernel launches, and the host-buffer convenience path.  No CPU fallback exists: without a CUDA
// device every entry point that needs one returns MACM_E_CUDA.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "macm_sim.h"

struct macm_sim {
    macm_params params;
    SimConst K;
    LaunchCfg cfg;
    int device;
    int bound;
    int blocks_per_sm, sm_count;
    int64_t launches;
    char cuda_err[256];
    // host-buffer path
    cudaStream_t hstream;
    void* d_actions;
    size_t d_actions_bytes;
    double2* d_sincos;
    int* d_scratch;            // two counters (macm_overflow_count)
    uint64_t auto_seed;        // seed of the resets appended under MACM_FLAG_AUTO_RESET
    Finals fin;                // macm_bind_final: where every reset copies the env's rows first
    // Ordering between the caller's streams and the handle's own host-path stream: the last stream an entry point
    // enqueued device work on, whether that work is still unordered against hstream, and the reverse.  Events are
    // recorded lazily, at the moment the other side is used -- nothing is inserted between two step launches
    // (an event between them would end their programmatic overlap).
    cudaStream_t last_stream;
    int dev_dirty, host_dirty;
    cudaEvent_t ev_dev, ev_host;
};

// Every entry point that launches or allocates runs with the handle's device current and puts the caller's device
// back on return (a handle may be driven from a thread whose current device is another GPU).
struct DevGuard {
    int prev;
    bool ok;
    explicit DevGuard(int device) : prev(-1), ok(true)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != device) ok = cudaSetDevice(device) == cudaSuccess;
    }
    ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

static int fail_cuda(macm_sim* s, cudaError_t e, const char* where)
{
    if (s) snprintf(s->cuda_err, sizeof(s->cuda_err), "%s: %s", where, cudaGetErrorString(e));
    return MACM_E_CUDA;
}
#define CU(call)                                                   \
    do {                                                           \
        cudaError_t e_ = (call);                                   \
        if (e_ != cudaSuccess) return fail_cuda(sim, e_, #call);   \
    } while (0)

#define GUARD()                                                                  \
    DevGuard guard_(sim->device);                                                \
    if (!guard_.ok) return fail_cuda(sim, cudaGetLastError(), "cudaSetDevice")

// device work was enqueued on `s` by a caller-stream entry point
static void note_device_work(macm_sim* sim, cudaStream_t s) { sim->last_stream = s; sim->dev_dirty = 1; }

// `s` (a caller's stream) is about to touch the bound buffers: order it after whatever the host path enqueued
static int order_after_host(macm_sim* sim, cudaStream_t s)
{
    if (sim->host_dirty && sim->hstream) {
        CU(cudaEventRecord(sim->ev_host, sim->hstream));
        CU(cudaStreamWaitEvent(s, sim->ev_host, 0));
        sim->host_dirty = 0;
    }
    return MACM_OK;
}

// the host path is about to touch the bound buffers: order hstream after the caller-stream work seen so far
static int order_after_device(macm_sim* sim)
{
    if (sim->dev_dirty) {
        CU(cudaEventRecord(sim->ev_dev, sim->last_stream));
        CU(cudaStreamWaitEvent(sim->hstream, sim->ev_dev, 0));
        sim->dev_dirty = 0;
    }
    return MACM_OK;
}

static SampleConst sample_const(const macm_sim* sim, uint64_t seed)
{
    const macm_params& p = sim->params;
    SampleConst sc;
    sc.seed = seed; sc.spread = p.start_spread; sc.sx = p.start_x; sc.sy = p.start_y;
    sc.tmin = p.target_mindist; sc.tmax = p.target_maxdist; sc.width = p.world_width; sc.height = p.world_height;
    return sc;
}

// MACM_FLAG_AUTO_RESET: the launch that follows every step / rollout launch.  `row`: the last row of a rollout's
// final_* arrays, which receives the terminal rows of the envs this launch restarts
static int auto_reset(macm_sim* sim, cudaStream_t s, const Finals& row = Finals{})
{
    if (!(sim->params.flags & MACM_FLAG_AUTO_RESET)) return MACM_OK;
    CU(macm_launch_reset_masked(sim->K, sim->cfg, nullptr, sample_const(sim, sim->auto_seed), sim->fin, row, s));
    sim->launches += 1;
    return MACM_OK;
}

extern "C" int macm_abi_version(void) { return MACM_ABI_VERSION; }

extern "C" const char* macm_strerror(int status)
{
    switch (status) {
        case MACM_OK: return "ok";
        case MACM_E_INVALID: return "invalid argument";
        case MACM_E_CUDA: return "CUDA error (see macm_last_cuda_error)";
        case MACM_E_UNBOUND: return "buffers not bound";
        case MACM_E_ALIGN: return "buffer misaligned";
        case MACM_E_NOMEM: return "out of memory";
        case MACM_E_UNSUPPORTED: return "unsupported";
        default: return "unknown status";
    }
}

extern "C" const char* macm_last_cuda_error(const macm_sim* sim) { return sim ? sim->cuda_err : ""; }

extern "C" int macm_params_default(macm_params* p, int env_kind)
{
    if (!p || (env_kind != MACM_ENV_FLOCK && env_kind != MACM_ENV_TDM)) return MACM_E_INVALID;
    memset(p, 0, sizeof(*p));
    p->env_kind = env_kind;
    p->n_envs = 1;
    p->n_agents = env_kind == MACM_ENV_FLOCK ? 10 : 2;   // mvmnt.py:35, combat.py:61
    p->n_targets = env_kind == MACM_ENV_FLOCK ? 1 : 0;
    p->hz = 60.0;
    p->velocity_iterations = 8;
    p->position_iterations = 3;
    p->warm_starting = 1;
    p->damping_model = MACM_DAMPING_PADE;   // pip pybox2d bundles Box2D >= 2.3.1 (see gym_macm/settings.py)
    p->radius = 0.5;
    p->density = 1.0;
    p->friction = 0.3;
    p->linear_damping = 5.0;
    p->agent_force = 20.0;
    p->agent_rotation_speed = 0.8 * (2 * NP_PI);
    p->time_limit = 60.0;
    p->reward_mode = MACM_REWARD_BINARY;
    p->action_mode = MACM_ACTION_DISCRETE;
    p->coord = MACM_COORD_POLAR;
    p->flags = MACM_FLAG_REPAIR_MOV_COOLDOWN;
    p->reward_radius = 7.0;
    p->cooldown_atk = 1.0;
    p->cooldown_mov_penalty = 0.5;
    p->melee_range = 2.0;
    p->melee_dmg = 0.25;
    p->percent_mov_penalty = 0.2;
    p->init_health = 1.0;
    p->start_spread = 20.0;
    p->start_x = 0.0;
    p->start_y = 0.0;
    p->target_mindist = 25.0;
    p->target_maxdist = 60.0;
    p->world_width = 30.0;
    p->world_height = 30.0;
    return MACM_OK;
}

// number of `c -= 1/hz` float64 decrements until c <= 0 (combat.py:142,155)
static int cooldown_steps(double c, double hz)
{
    int k = 0;
    while (c > 0 && k < (1 << 24)) { c -= (1 / hz); ++k; }
    return k;
}

static int derive_constants(macm_sim* sim)
{
    const macm_params& p = sim->params;
    SimConst& K = sim->K;
    memset(&K, 0, sizeof(K));
    K.E = p.n_envs; K.N = p.n_agents; K.T = p.n_targets;
    K.env_base = p.env_index_base;
    const int pairs = p.n_agents * (p.n_agents - 1) / 2;
    int C = p.max_contacts > 0 ? p.max_contacts : (pairs < 8 * p.n_agents ? pairs : 8 * p.n_agents);
    if (C > pairs) C = pairs;
    if (C < 1) C = 1;
    int TC = p.max_touching > 0 ? p.max_touching : (C < 2 * p.n_agents ? C : 2 * p.n_agents);
    if (TC > C) TC = C;
    // envs of 65..128 agents: the default leaves room for one 448-thread block (14 envs) per SM in shared memory
    if (p.max_touching <= 0 && p.n_agents > 64 && TC > 192) TC = 192;
    TC = (TC + 15) / 16 * 16;
    // macm_rollout parks 20 bytes per agent slot in the (24-byte-per-entry) touching-contact stage between steps
    {
        const int slots = p.n_agents > 64 ? 128 : (p.n_agents > 32 ? 64 : (p.n_agents > 16 ? 32 : 16));
        const int need = (20 * slots + 23) / 24;
        if (TC < need) TC = (need + 15) / 16 * 16;
    }
    int TCH = 0;             // beyond the shared-memory stage: a global-memory one of the requested capacity
    if (TC > 240) { TCH = (TC + 7) / 8 * 8; TC = 240; }  // (shared-memory stage: levels and list links are bytes)
    // envs of 65..128 agents by default: a gathered flock (the bots.flock actor at the target) reaches up to ~1.8N
    // touching contacts, more than the 192 of the shared stage from about 116 agents on, so a global-memory stage of
    // 3N takes what the shared one cannot hold
    if (p.max_touching <= 0 && p.n_agents > 64) {
        const int h = C < 3 * p.n_agents ? C : 3 * p.n_agents;
        if (h > TC) TCH = (h + 7) / 8 * 8;
    }
    K.C = C; K.TC = TC; K.TCH = TCH;
    K.kind = p.env_kind; K.reward_mode = p.reward_mode; K.action_mode = p.action_mode; K.coord = p.coord;
    K.vel_iters = p.velocity_iterations; K.pos_iters = p.position_iterations;
    K.warm_starting = p.warm_starting; K.flags = p.flags;
    K.obs_dim = p.env_kind == MACM_ENV_TDM ? 4 * p.n_agents : (p.coord == MACM_COORD_POLAR ? 4 : 6);
    K.obs_dtype = p.obs_dtype;
    K.obs_words = p.obs_dtype == MACM_OBS_F32 ? K.obs_dim : K.obs_dim / 2;   // obs_dim is even

    // cm_framework.py:182,222: timeStep = 1.0/hz is a Python float, rounded to float32 by SWIG
    K.h = (float)(1.0 / p.hz);
    const float inv_dt = 1.0f / K.h;          // b2World::Step: step.inv_dt
    K.dt_ratio = inv_dt * K.h;                // m_inv_dt0 * dt from the second step on
    K.radius = (float)p.radius;
    const float mass = (float)p.density * B2_PI * K.radius * K.radius;  // b2CircleShape::ComputeMass
    K.inv_mass = 1.0f / mass;
    const float fr = (float)p.friction;
    K.friction = sqrtf(fr * fr);              // b2MixFriction
    const float ld = (float)p.linear_damping;
    if (p.damping_model == MACM_DAMPING_TAYLOR) {
        float d = 1.0f - K.h * ld;
        K.damp = d < 0.0f ? 0.0f : (d > 1.0f ? 1.0f : d);
    } else {
        K.damp = 1.0f / (1.0f + K.h * ld);
    }
    const float rsum = K.radius + K.radius;
    K.rsum2 = rsum * rsum;
    K.k_sum = K.inv_mass + K.inv_mass;
    K.normal_mass = K.k_sum > 0.0f ? 1.0f / K.k_sum : 0.0f;

    // binary reward: int(sqrt64(d2_f32) < reward_radius)  <=>  d2_f32 < thr  (sqrt is monotone)
    {
        const double R = p.reward_radius;
        float x = (float)(R * R);
        if (!(R > 0)) x = 0.0f;
        else {
            while (sqrt((double)x) < R) x = nextafterf(x, INFINITY);
            while (x > 0.0f && !(sqrt((double)nextafterf(x, -INFINITY)) < R)) x = nextafterf(x, -INFINITY);
        }
        K.binary_thr = x;
    }
    // done = (time_passed > time_limit) with time_passed accumulated in float64 (mvmnt.py:134-136)
    {
        double t = 0.0;
        int k = 0;
        const int cap = 1 << 28;
        while (k < cap) { t += (1 / p.hz); ++k; if (t > p.time_limit) break; }
        K.done_step = k < cap ? k : 0x7fffffff;
    }
    K.rot_step = p.agent_rotation_speed * (1 / p.hz);
    K.force = p.agent_force;
    K.force_pen = p.agent_force * (1 - p.percent_mov_penalty * 1);
    K.diag = 1 / sqrt(2.0);
    K.melee_range = p.melee_range;
    K.melee_dmg = (float)p.melee_dmg;
    K.melee_dmg_d = p.melee_dmg;
    K.init_health = (float)p.init_health;
    K.cd_atk_steps = cooldown_steps(p.cooldown_atk, p.hz);
    K.cd_mov_steps = cooldown_steps(p.cooldown_mov_penalty, p.hz);
    return MACM_OK;
}

extern "C" int macm_create(macm_sim** out, const macm_params* p, int device)
{
    if (!out || !p) return MACM_E_INVALID;
    *out = nullptr;
    if (p->env_kind != MACM_ENV_FLOCK && p->env_kind != MACM_ENV_TDM) return MACM_E_INVALID;
    if (p->n_envs < 1 || p->n_agents < 2 || p->n_agents > MACM_MAX_AGENTS) return MACM_E_INVALID;
    if (p->env_kind == MACM_ENV_FLOCK && (p->n_targets < 1 || p->n_targets > MACM_MAX_TARGETS)) return MACM_E_INVALID;
    if (!(p->hz > 0) || !(p->radius > 0) || !(p->density > 0) || p->friction < 0 || p->linear_damping < 0)
        return MACM_E_INVALID;
    if (p->velocity_iterations < 0 || p->position_iterations < 0) return MACM_E_INVALID;
    if (p->reward_mode < 0 || p->reward_mode > 1 || p->action_mode < 0 || p->action_mode > 1 || p->coord < 0 ||
        p->coord > 1 || p->damping_model < 0 || p->damping_model > 1)
        return MACM_E_INVALID;
    if (p->obs_dtype != MACM_OBS_F32 && p->obs_dtype != MACM_OBS_F16 && p->obs_dtype != MACM_OBS_BF16) return MACM_E_INVALID;

    macm_sim* sim = new (std::nothrow) macm_sim;
    if (!sim) return MACM_E_NOMEM;
    memset(sim, 0, sizeof(*sim));
    sim->params = *p;
    sim->device = device;
    int rc = derive_constants(sim);
    if (rc != MACM_OK) { delete sim; return rc; }

    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
        // report through a static string: the handle is not returned
        delete sim;
        return MACM_E_CUDA;
    }
    // the handle is returned even when a CUDA call below fails, so that macm_last_cuda_error can say why;
    // the caller destroys it (macm_destroy frees whatever was allocated)
    *out = sim;
    GUARD();
    CU(cudaDeviceGetAttribute(&sim->sm_count, cudaDevAttrMultiProcessorCount, device));
    e = macm_launch_cfg(sim->K, sim->sm_count, &sim->cfg);
    if (e != cudaSuccess) { *out = nullptr; delete sim; return MACM_E_INVALID; }
    CU(macm_prepare_kernels(sim->K, sim->cfg, &sim->blocks_per_sm));
    if (sim->K.TCH > 0) CU(macm_prepare_kernels_huge(sim->K, sim->cfg));
    sim->K.first_wave = sim->sm_count * (sim->blocks_per_sm > 0 ? sim->blocks_per_sm : 1);
    // sin/cos(k/128), k = 0..417, as float64: the table behind the action decode's np.cos/np.sin
    {
        const int n = 418;
        double2 tab[n];
        for (int k = 0; k < n; ++k) { tab[k].x = sin(k * 0.0078125); tab[k].y = cos(k * 0.0078125); }
        CU(cudaMalloc((void**)&sim->d_sincos, sizeof(tab)));
        CU(cudaMemcpy(sim->d_sincos, tab, sizeof(tab), cudaMemcpyHostToDevice));
        sim->K.sincos_tab = sim->d_sincos;
    }
    CU(cudaMalloc((void**)&sim->d_scratch, 2 * sizeof(int)));
    CU(cudaEventCreateWithFlags(&sim->ev_dev, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&sim->ev_host, cudaEventDisableTiming));
    return MACM_OK;
}

extern "C" int macm_destroy(macm_sim* sim)
{
    if (!sim) return MACM_E_INVALID;
    {
        DevGuard guard_(sim->device);
        if (sim->d_actions) cudaFree(sim->d_actions);
        if (sim->d_sincos) cudaFree(sim->d_sincos);
        if (sim->d_scratch) cudaFree(sim->d_scratch);
        if (sim->ev_dev) cudaEventDestroy(sim->ev_dev);
        if (sim->ev_host) cudaEventDestroy(sim->ev_host);
        if (sim->hstream) cudaStreamDestroy(sim->hstream);
    }
    delete sim;
    return MACM_OK;
}

extern "C" int macm_get_buffer_sizes(const macm_sim* sim, macm_buffer_sizes* o)
{
    if (!sim || !o) return MACM_E_INVALID;
    memset(o, 0, sizeof(*o));
    const SimConst& K = sim->K;
    const uint64_t EN = (uint64_t)K.E * K.N;
    o->posvel = EN * 16; o->angsleep = EN * 8; o->fat = EN * 16;
    o->contact_ab = (uint64_t)K.E * K.C * 4; o->contact_imp = (uint64_t)K.E * K.C * 8;
    o->contact_count = (uint64_t)K.E * 4; o->env_state = (uint64_t)K.E * 16;
    o->targets = (uint64_t)K.E * K.T * 8; o->target_idx = K.kind == MACM_ENV_FLOCK ? (uint64_t)K.N : 0;
    o->tdm_state = K.kind == MACM_ENV_TDM ? EN * 16 : 0; o->team = K.kind == MACM_ENV_TDM ? (uint64_t)K.N : 0;
    o->obs = EN * 4 * (uint64_t)K.obs_words; o->nn_idx = K.kind == MACM_ENV_FLOCK ? EN * 4 : 0;
    o->rewards = EN * 4; o->collided = EN; o->done = (uint64_t)K.E;
    o->touch_scratch = (uint64_t)K.E * K.TCH * 32;
    o->obs_dim = K.obs_dim;
    o->action_bytes = sim->params.action_mode == MACM_ACTION_DISCRETE ? 4 : 8;
    o->max_contacts = K.C; o->max_touching = K.TCH > 0 ? K.TCH : K.TC;
    return MACM_OK;
}

extern "C" int macm_get_launch_info(const macm_sim* sim, macm_launch_info* o)
{
    if (!sim || !o) return MACM_E_INVALID;
    o->lanes_per_env = sim->cfg.G; o->agents_per_lane = sim->cfg.APL; o->envs_per_block = sim->cfg.envs_per_block;
    o->threads_per_block = sim->cfg.threads; o->blocks = sim->cfg.blocks; o->smem_bytes_per_block = sim->cfg.smem_bytes;
    o->blocks_per_sm = sim->blocks_per_sm; o->sm_count = sim->sm_count; o->done_step = sim->K.done_step;
    o->dt = sim->K.h; o->dt_ratio = sim->K.dt_ratio; o->inv_mass = sim->K.inv_mass; o->damping_factor = sim->K.damp;
    o->binary_d2_threshold = sim->K.binary_thr;
    return MACM_OK;
}

static bool aligned(const void* p, size_t a) { return ((uintptr_t)p % a) == 0; }

// alignment of an observation array: the vector width of its record stores -- float4 in fp32, one 8-byte record of
// four 16-bit values (Flock polar, TDM), or three 32-bit words (Flock cartesian, 12-byte records)
static size_t obs_align(const SimConst& K)
{
    if (K.obs_dtype == MACM_OBS_F32) return 16;
    return (K.kind == MACM_ENV_FLOCK && K.coord == MACM_COORD_CARTESIAN) ? 4 : 8;
}

extern "C" int macm_bind(macm_sim* sim, const macm_buffers* b)
{
    if (!sim || !b) return MACM_E_INVALID;
    SimConst& K = sim->K;
    const bool flock = K.kind == MACM_ENV_FLOCK;
    if (!b->posvel || !b->angsleep || !b->fat || !b->contact_ab || !b->contact_imp || !b->contact_count ||
        !b->env_state || !b->obs || !b->rewards || !b->collided || !b->done)
        return MACM_E_UNBOUND;
    if (flock && (!b->targets || !b->target_idx || !b->nn_idx)) return MACM_E_UNBOUND;
    if (!flock && (!b->tdm_state || !b->team)) return MACM_E_UNBOUND;
    if (!aligned(b->posvel, 16) || !aligned(b->fat, 16) || !aligned(b->angsleep, 8) || !aligned(b->contact_imp, 8) ||
        !aligned(b->contact_ab, 4) || !aligned(b->env_state, 16) || !aligned(b->obs, obs_align(K)) || !aligned(b->rewards, 4) ||
        (b->targets && !aligned(b->targets, 8)) || (b->tdm_state && !aligned(b->tdm_state, 16)) ||
        (b->nn_idx && !aligned(b->nn_idx, 4)))
        return MACM_E_ALIGN;
    K.posvel = (float4*)b->posvel; K.angsleep = (float2*)b->angsleep; K.fat = (float4*)b->fat;
    K.c_ab = b->contact_ab; K.c_imp = (float2*)b->contact_imp; K.c_cnt = b->contact_count;
    K.env_state = (int4*)b->env_state; K.targets = (const float2*)b->targets; K.target_idx = b->target_idx;
    K.tdm = (float4*)b->tdm_state; K.team = b->team;
    K.obs = b->obs; K.nn_idx = b->nn_idx; K.rewards = b->rewards; K.collided = b->collided; K.done = b->done;
    if (K.TCH > 0 && (!b->touch_scratch || !aligned(b->touch_scratch, 16))) return b->touch_scratch ? MACM_E_ALIGN : MACM_E_UNBOUND;
    K.scratch = K.TCH > 0 ? b->touch_scratch : nullptr;
    sim->bound = 1;
    return MACM_OK;
}

// the final arrays of `f` fit this sim's env kind and the alignment of the bound buffers of the same names
static int check_final(const macm_sim* sim, const float* obs, const int32_t* nn_idx, const float* tdm_state,
                       const int32_t* env_state)
{
    const bool flock = sim->K.kind == MACM_ENV_FLOCK;
    if ((nn_idx && !flock) || (tdm_state && flock)) return MACM_E_INVALID;
    if ((obs && !aligned(obs, obs_align(sim->K))) || (nn_idx && !aligned(nn_idx, 4)) || (tdm_state && !aligned(tdm_state, 16)) ||
        (env_state && !aligned(env_state, 16)))
        return MACM_E_ALIGN;
    return MACM_OK;
}

extern "C" int macm_bind_final(macm_sim* sim, const macm_final_out* f)
{
    if (!sim) return MACM_E_INVALID;
    if (!f) { sim->fin = Finals{}; return MACM_OK; }
    if (int rc = check_final(sim, f->obs, f->nn_idx, f->tdm_state, f->env_state)) return rc;
    sim->fin = Finals{f->obs, f->nn_idx, (float4*)f->tdm_state, (int4*)f->env_state};
    return MACM_OK;
}

extern "C" int macm_reset(macm_sim* sim, void* stream)
{
    if (!sim) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    CU(macm_launch_reset(sim->K, (cudaStream_t)stream));
    CU(macm_launch_observe(sim->K, sim->cfg, (cudaStream_t)stream));
    sim->launches += 2;
    note_device_work(sim, (cudaStream_t)stream);
    return MACM_OK;
}

extern "C" int macm_sample_reset(macm_sim* sim, uint64_t seed, void* stream)
{
    if (!sim) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    CU(macm_launch_sample(sim->K, sample_const(sim, seed), (cudaStream_t)stream));
    sim->launches += 1;
    return macm_reset(sim, stream);
}

extern "C" int macm_reset_masked(macm_sim* sim, const uint8_t* mask, uint64_t seed, void* stream)
{
    if (!sim) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    CU(macm_launch_reset_masked(sim->K, sim->cfg, mask, sample_const(sim, seed), sim->fin, Finals{}, (cudaStream_t)stream));
    sim->launches += 1;
    note_device_work(sim, (cudaStream_t)stream);
    return MACM_OK;
}

extern "C" int macm_set_auto_reset_seed(macm_sim* sim, uint64_t seed)
{
    if (!sim) return MACM_E_INVALID;
    sim->auto_seed = seed;
    return MACM_OK;
}

extern "C" int macm_overflow_count(macm_sim* sim, int32_t* contact_envs, int32_t* touching_envs, void* stream)
{
    if (!sim) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    CU(macm_launch_overflow_count(sim->K, sim->d_scratch, (cudaStream_t)stream));
    sim->launches += 1;
    int h[2] = {0, 0};
    CU(cudaMemcpyAsync(h, sim->d_scratch, sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    if (contact_envs) *contact_envs = h[0];
    if (touching_envs) *touching_envs = h[1];
    return MACM_OK;
}

extern "C" int macm_pack_actions(macm_sim* sim, const void* src, int32_t elem_bytes, int32_t width, void* actions_out,
                                 void* stream)
{
    if (!sim || !src || !actions_out) return MACM_E_INVALID;
    if ((elem_bytes != 1 && elem_bytes != 2 && elem_bytes != 4 && elem_bytes != 8) || (width != 3 && width != 4))
        return MACM_E_INVALID;
    if (!aligned(actions_out, 4)) return MACM_E_ALIGN;
    GUARD();
    CU(macm_launch_pack_actions(src, elem_bytes, width, (uint64_t)sim->K.E * sim->K.N, actions_out, (cudaStream_t)stream));
    sim->launches += 1;
    return MACM_OK;
}

extern "C" int macm_step(macm_sim* sim, const void* actions, void* stream)
{
    if (!sim || !actions) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    if (!aligned(actions, sim->params.action_mode == MACM_ACTION_DISCRETE ? 4 : 8)) return MACM_E_ALIGN;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    Rollout R = {};
    R.K = 1;
    R.policy = -1;
    CU(macm_launch_step(sim->K, sim->cfg, actions, R, (cudaStream_t)stream));
    sim->launches += 1;
    note_device_work(sim, (cudaStream_t)stream);
    return auto_reset(sim, (cudaStream_t)stream);
}

extern "C" int macm_rollout(macm_sim* sim, const void* actions, int32_t n_steps, int32_t policy, uint64_t seed,
                            const macm_rollout_out* out, void* stream)
{
    if (!sim || n_steps < 1) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    const bool discrete = sim->params.action_mode == MACM_ACTION_DISCRETE;
    Rollout R = {};
    R.K = n_steps;
    R.policy = -1;
    R.seed = seed;
    R.sc = sample_const(sim, sim->auto_seed);
    R.sync = sim->cfg.threads > 128 ? 1 : 0;   // wide blocks: the warps of a block run each step in step
    if (const char* e = getenv("MACM_ROLLOUT_SYNC")) R.sync = atoi(e);   // experiments
    if (actions) {
        if (!aligned(actions, discrete ? 4 : 8)) return MACM_E_ALIGN;
    } else {
        // actions=None: every agent's actor decides from its own observation (mvmnt.py:86-92)
        if (policy < MACM_BOT_IDLE || policy > MACM_BOT_CIRCLE) return MACM_E_INVALID;
        if (!discrete) return MACM_E_UNSUPPORTED;
        if (policy == MACM_BOT_FLOCK && (sim->K.kind != MACM_ENV_FLOCK || sim->params.coord != MACM_COORD_POLAR))
            return MACM_E_UNSUPPORTED;
        // the flock actor's first step reads the stored observation: a rounded one would change its decisions
        if (policy == MACM_BOT_FLOCK && sim->K.obs_dtype != MACM_OBS_F32) return MACM_E_UNSUPPORTED;
        if (policy == MACM_BOT_COMBAT && sim->K.kind != MACM_ENV_TDM) return MACM_E_UNSUPPORTED;
        R.policy = policy;
    }
    if (out) {
        if ((out->obs && !aligned(out->obs, obs_align(sim->K))) || (out->rewards && !aligned(out->rewards, 4)) ||
            (out->nn_idx && !aligned(out->nn_idx, 4)))
            return MACM_E_ALIGN;
        R.obs = out->obs; R.nn_idx = out->nn_idx; R.rewards = out->rewards; R.collided = out->collided; R.done = out->done;
        if (int rc = check_final(sim, out->final_obs, out->final_nn_idx, out->final_tdm_state, out->final_env_state))
            return rc;
        R.fin_k = Finals{out->final_obs, out->final_nn_idx, (float4*)out->final_tdm_state, (int4*)out->final_env_state};
    }
    R.fin = sim->fin;
    R.finals = R.fin.obs || R.fin.nn_idx || R.fin.tdm || R.fin.es || R.fin_k.obs || R.fin_k.nn_idx || R.fin_k.tdm ||
               R.fin_k.es;
    // the launch's last step: the appended reset copies its terminal rows to row n_steps - 1 of the final_* arrays
    const SimConst& K = sim->K;
    const size_t last = (size_t)(n_steps - 1) * K.E, EN = last * K.N;
    const Finals row = {R.fin_k.obs ? R.fin_k.obs + EN * K.obs_words : nullptr, R.fin_k.nn_idx ? R.fin_k.nn_idx + EN : nullptr,
                        R.fin_k.tdm ? R.fin_k.tdm + EN : nullptr, R.fin_k.es ? R.fin_k.es + last : nullptr};
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    CU(macm_launch_step(sim->K, sim->cfg, actions, R, (cudaStream_t)stream));
    sim->launches += 1;
    note_device_work(sim, (cudaStream_t)stream);
    return auto_reset(sim, (cudaStream_t)stream, row);
}

extern "C" int macm_observe(macm_sim* sim, void* stream)
{
    if (!sim) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    CU(macm_launch_observe(sim->K, sim->cfg, (cudaStream_t)stream));
    sim->launches += 1;
    note_device_work(sim, (cudaStream_t)stream);
    return MACM_OK;
}

extern "C" int macm_bot_actions(macm_sim* sim, int policy, uint64_t seed, void* actions_out, void* stream)
{
    if (!sim || !actions_out) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    if (policy < MACM_BOT_IDLE || policy > MACM_BOT_CIRCLE) return MACM_E_INVALID;
    if (sim->params.action_mode != MACM_ACTION_DISCRETE) return MACM_E_UNSUPPORTED;
    if (policy == MACM_BOT_COMBAT && sim->K.kind != MACM_ENV_TDM) return MACM_E_UNSUPPORTED;
    if (policy == MACM_BOT_FLOCK && sim->K.kind != MACM_ENV_FLOCK) return MACM_E_UNSUPPORTED;
    // these two actors decide from the stored observation: a rounded one would change their decisions
    if ((policy == MACM_BOT_FLOCK || policy == MACM_BOT_COMBAT) && sim->K.obs_dtype != MACM_OBS_F32)
        return MACM_E_UNSUPPORTED;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    CU(macm_launch_bot(sim->K, policy, seed, actions_out, (cudaStream_t)stream));
    sim->launches += 1;
    return MACM_OK;
}

extern "C" int macm_render(macm_sim* sim, const macm_render_args* a, void* stream)
{
    if (!sim || !a) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    if (a->n_frames < 1 || a->height < 1 || a->height > 4096 || a->width < 1 || a->width > 4096) return MACM_E_INVALID;
    if (!a->views || !a->palette || !a->out || (!a->envs && a->n_frames > sim->K.E)) return MACM_E_INVALID;
    if (!aligned(a->views, 4) || (a->envs && !aligned(a->envs, 4))) return MACM_E_ALIGN;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    const SimConst& K = sim->K;
    const bool flock = K.kind == MACM_ENV_FLOCK;
    const RenderConst R = {K.E, K.N, flock ? K.T : 0, K.kind, sim->params.radius, sim->params.reward_radius,
                           K.posvel, K.angsleep, K.collided, K.tdm, K.targets};
    CU(macm_launch_render(R, *a, (cudaStream_t)stream));
    sim->launches += 1;
    note_device_work(sim, (cudaStream_t)stream);   // the host path must not overwrite the state before it is drawn
    return MACM_OK;
}

extern "C" int macm_render_agents(macm_sim* sim, const macm_agent_frames_args* a, void* stream)
{
    if (!sim || !a) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    if (a->n_envs < 1 || a->height < 1 || a->height > 1024 || a->width < 1 || a->width > 1024) return MACM_E_INVALID;
    if (!(a->half_width > 0.0 && isfinite(a->half_width))) return MACM_E_INVALID;
    if (!a->palette || !a->out || (!a->envs && a->n_envs > sim->K.E)) return MACM_E_INVALID;
    if (a->envs && !aligned(a->envs, 4)) return MACM_E_ALIGN;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    const SimConst& K = sim->K;
    const bool flock = K.kind == MACM_ENV_FLOCK;
    const RenderConst R = {K.E, K.N, flock ? K.T : 0, K.kind, sim->params.radius, sim->params.reward_radius,
                           K.posvel, K.angsleep, K.collided, K.tdm, K.targets};
    CU(macm_launch_render_agents(R, *a, (cudaStream_t)stream));
    sim->launches += 1;
    note_device_work(sim, (cudaStream_t)stream);   // the host path must not overwrite the state before it is drawn
    return MACM_OK;
}

extern "C" int macm_lidar(macm_sim* sim, const macm_lidar_args* a, void* stream)
{
    if (!sim || !a) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    if (a->n_envs < 1 || a->n_rays < 1 || a->n_rays > MACM_MAX_RAYS) return MACM_E_INVALID;
    if (!(isfinite(a->max_range) && a->max_range > 0.0 && a->max_range <= 1e6)) return MACM_E_INVALID;
    if (!(isfinite(a->fov) && a->fov > 0.0 && a->fov <= 2.0 * NP_PI)) return MACM_E_INVALID;
    if (!a->fraction || (!a->envs && a->n_envs > sim->K.E)) return MACM_E_INVALID;
    const SimConst& K = sim->K;
    if ((a->envs && !aligned(a->envs, 4)) || (a->hit && !aligned(a->hit, 4)) ||
        !aligned(a->fraction, K.obs_dtype == MACM_OBS_F32 ? 4 : 2))
        return MACM_E_ALIGN;
    GUARD();
    if (int rc = order_after_host(sim, (cudaStream_t)stream)) return rc;
    const RenderConst R = {K.E, K.N, K.kind == MACM_ENV_FLOCK ? K.T : 0, K.kind, sim->params.radius,
                           sim->params.reward_radius, K.posvel, K.angsleep, K.collided, K.tdm, K.targets};
    CU(macm_launch_lidar(R, *a, K.obs_dtype, (cudaStream_t)stream));
    sim->launches += 1;
    note_device_work(sim, (cudaStream_t)stream);   // the host path must not overwrite the state before it is scanned
    return MACM_OK;
}

extern "C" int macm_step_host_async(macm_sim* sim, const void* actions, float* obs, float* rewards, int32_t* nn_idx,
                                    uint8_t* collided, uint8_t* done)
{
    if (!sim || !actions) return MACM_E_INVALID;
    if (!sim->bound) return MACM_E_UNBOUND;
    GUARD();
    macm_buffer_sizes z;
    macm_get_buffer_sizes(sim, &z);
    const size_t abytes = (size_t)sim->K.E * sim->K.N * z.action_bytes;
    if (!sim->hstream) CU(cudaStreamCreateWithFlags(&sim->hstream, cudaStreamNonBlocking));
    if (sim->d_actions_bytes < abytes) {
        if (sim->d_actions) cudaFree(sim->d_actions);
        sim->d_actions = nullptr;
        sim->d_actions_bytes = 0;
        CU(cudaMalloc(&sim->d_actions, abytes));
        sim->d_actions_bytes = abytes;
    }
    cudaStream_t s = sim->hstream;
    // resets, steps, state loads enqueued on the caller's streams so far come first
    if (int rc = order_after_device(sim)) return rc;
    CU(cudaMemcpyAsync(sim->d_actions, actions, abytes, cudaMemcpyHostToDevice, s));
    Rollout R = {};
    R.K = 1;
    R.policy = -1;
    CU(macm_launch_step(sim->K, sim->cfg, sim->d_actions, R, s));
    sim->launches += 1;
    if (int rc = auto_reset(sim, s)) return rc;   // before the copies: a finished env reports its new episode's first observation
    // Device -> host: one DMA per run of outputs that is contiguous on BOTH sides (the host package lays the
    // five output arrays out back to back in one device slab and one pinned slab, so a step's results travel
    // in a single transfer -- SURVEY 8(f1): "one D2H"); separate arrays still get a copy each.
    struct Seg { char* dst; const char* src; size_t n; };
    Seg seg[5];
    int ns = 0;
    if (obs) seg[ns++] = {(char*)obs, (const char*)sim->K.obs, (size_t)z.obs};
    if (rewards) seg[ns++] = {(char*)rewards, (const char*)sim->K.rewards, (size_t)z.rewards};
    if (nn_idx && sim->K.nn_idx) seg[ns++] = {(char*)nn_idx, (const char*)sim->K.nn_idx, (size_t)z.nn_idx};
    if (collided) seg[ns++] = {(char*)collided, (const char*)sim->K.collided, (size_t)z.collided};
    if (done) seg[ns++] = {(char*)done, (const char*)sim->K.done, (size_t)z.done};
    for (int i = 1; i < ns; ++i)   // by device address
        for (int j = i; j > 0 && seg[j].src < seg[j - 1].src; --j) { Seg t = seg[j]; seg[j] = seg[j - 1]; seg[j - 1] = t; }
    for (int i = 0; i < ns;) {
        size_t n = seg[i].n;
        int j = i + 1;
        // the next array starts within 256 bytes of this one's end (alignment padding) at the same offset on both sides
        while (j < ns && seg[j].src >= seg[i].src + n && seg[j].src - (seg[i].src + n) < 256 &&
               seg[j].dst - seg[i].dst == seg[j].src - seg[i].src) {
            n = (size_t)(seg[j].src - seg[i].src) + seg[j].n;
            ++j;
        }
        CU(cudaMemcpyAsync(seg[i].dst, seg[i].src, n, cudaMemcpyDeviceToHost, s));
        i = j;
    }
    sim->host_dirty = 1;
    return MACM_OK;
}

extern "C" int macm_host_sync(macm_sim* sim)
{
    if (!sim) return MACM_E_INVALID;
    if (sim->hstream) CU(cudaStreamSynchronize(sim->hstream));
    sim->host_dirty = 0;
    return MACM_OK;
}

extern "C" int macm_step_host(macm_sim* sim, const void* actions, float* obs, float* rewards, int32_t* nn_idx,
                              uint8_t* collided, uint8_t* done)
{
    const int rc = macm_step_host_async(sim, actions, obs, rewards, nn_idx, collided, done);
    return rc != MACM_OK ? rc : macm_host_sync(sim);
}

extern "C" int macm_host_alloc(void** out, uint64_t bytes)
{
    if (!out) return MACM_E_INVALID;
    return cudaMallocHost(out, bytes) == cudaSuccess ? MACM_OK : MACM_E_CUDA;
}

extern "C" int macm_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? MACM_OK : MACM_E_CUDA; }

extern "C" int macm_enable_peer_access(int device, int peer_device)
{
    if (device == peer_device) return MACM_OK;
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, device, peer_device) != cudaSuccess || !can) return MACM_E_UNSUPPORTED;
    int cur = 0;
    cudaGetDevice(&cur);
    if (cudaSetDevice(device) != cudaSuccess) return MACM_E_CUDA;
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
    cudaSetDevice(cur);
    return e == cudaSuccess ? MACM_OK : MACM_E_CUDA;
}

extern "C" int macm_device_alloc(int device, uint64_t bytes, void** out, void* ipc_handle_out)
{
    if (!out || bytes == 0) return MACM_E_INVALID;
    int cur = 0;
    cudaGetDevice(&cur);
    if (cudaSetDevice(device) != cudaSuccess) return MACM_E_CUDA;
    cudaError_t e = cudaMalloc(out, bytes);
    if (e == cudaSuccess) e = cudaMemset(*out, 0, bytes);
    if (e == cudaSuccess && ipc_handle_out) {
        cudaIpcMemHandle_t h;
        e = cudaIpcGetMemHandle(&h, *out);
        if (e == cudaSuccess) memcpy(ipc_handle_out, &h, sizeof(h));
    }
    if (e != cudaSuccess) { fprintf(stderr, "macm_device_alloc: %s\n", cudaGetErrorString(e)); cudaGetLastError(); }
    cudaSetDevice(cur);
    return e == cudaSuccess ? MACM_OK : MACM_E_CUDA;
}

extern "C" int macm_device_free(void* p) { return cudaFree(p) == cudaSuccess ? MACM_OK : MACM_E_CUDA; }

extern "C" int macm_ipc_open(const void* handle, int device, void** out)
{
    if (!handle || !out) return MACM_E_INVALID;
    int cur = 0;
    cudaGetDevice(&cur);
    if (cudaSetDevice(device) != cudaSuccess) return MACM_E_CUDA;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    // opened on the device whose kernels will use the mapping: peer access to the exporting GPU is set up with it
    cudaError_t e = cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { fprintf(stderr, "macm_ipc_open: %s\n", cudaGetErrorString(e)); cudaGetLastError(); }
    cudaSetDevice(cur);
    return e == cudaSuccess ? MACM_OK : MACM_E_CUDA;
}

extern "C" int macm_ipc_close(void* base) { return cudaIpcCloseMemHandle(base) == cudaSuccess ? MACM_OK : MACM_E_CUDA; }

extern "C" int macm_set_trace(macm_sim* sim, void* trace)
{
    if (!sim) return MACM_E_INVALID;
    if (trace && !aligned(trace, 8)) return MACM_E_ALIGN;
    sim->K.trace = (unsigned long long*)trace;
    return MACM_OK;
}

extern "C" int64_t macm_launch_count(const macm_sim* sim) { return sim ? sim->launches : 0; }
