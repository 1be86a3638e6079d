// macm_kernels.cu -- hand-written sm_100a kernels for the batched gym-macm step.
//
// One kernel launch == one Flock.step / TDM.step (mvmnt.py:81-140, combat.py:104-184) for every
// environment of the batch, i.e. action decode + b2World::Step + reward pass + observation pass.
//
// Mapping.  An environment is owned by a GROUP of G lanes of one warp (G = 4, 8, 16 or 32); each
// lane owns APL agents (agent i lives in lane i % G, slot i / G), so N <= G*APL <= 128.  Groups
// never talk to each other, so all synchronisation is __syncwarp / ballot on the group mask and
// a block is just a bag of independent groups (no __syncthreads anywhere).  The bodies, the fat
// AABBs, the contact adjacency (one 64- or 128-bit row per agent) and the touching contacts of an
// environment are staged in shared memory; HBM is touched once per array per step with
// coalesced float4 / float2 accesses.
//
// Exactness.  The engine arithmetic is Box2D's: fp32, round-to-nearest, NO fused multiply-add
// (this file is compiled with -fmad=false, IEEE division and square root), evaluated in the
// same association order as Box2D 2.3.0.  Contacts are solved in Box2D's island order: a
// depth-first traversal from the last-created body over contact edges newest-first.  Two
// contacts that share no body commute bit-exactly, so the ordered list is level-scheduled
// (level = 1 + max(level of the previous contact of either body)) and each level runs across
// lanes; contacts of the same level touch disjoint bodies.
//
// The reference's host arithmetic is Python float64 (angle update, sin/cos, force); that part is
// done in fp64 here and rounded to fp32 exactly where pybox2d's SWIG layer rounds.
#include <float.h>
#include <stdlib.h>

#include "macm_sim.h"

// macm_kernels_huge.cu compiles this file a second time with MACM_HUGE_TU defined: the same kernels plus the
// global-memory touching stage (max_touching > 240), exported as macm_launch_step_huge / macm_prepare_kernels_huge.
#ifdef MACM_HUGE_TU
#define MACM_HUGE_BUILD 1
#else
#define MACM_HUGE_BUILD 0
#endif

// Launch shapes: 128-thread blocks, 7 per SM (72 registers); or, for one-env-per-warp groups (N > 16),
// one 896-thread block per SM.  (Measured on B200, profiles/README.md: the
// warp scheduler favours the warps of the oldest resident block, so with seven small blocks the last
// block's warps only get the issue slots the others leave and an env with large islands in that
// block sets the kernel time; warps of one block are served evenly.)
#define MACM_WIDE_THREADS 896
#define MACM_TABLE_BYTES (418 * 16)   // sin/cos(k/128) as double2, staged per block in the wide launch

// Phase stamps for profiles/phase_trace.py (a separate build with -DMACM_PHASE_TRACE; the trace
// buffer then holds 16 words per env: SM clock at the end of each phase, relative to the start).
#ifdef MACM_PHASE_TRACE
#define PHASE_STAMP(k) do { g.sync(); if (P.trace && g.gl == 0) P.trace[(size_t)env * 16 + (k)] = clock64() - tr_c0; } while (0)
#else
#define PHASE_STAMP(k) do { } while (0)
#endif

namespace {

// Agent sets: one bit per agent of an env, agent i in bit i & 31 of word i >> 5 (slot s of a 32-lane group is word s).
// Two words for envs of up to 64 agents, four beyond; a set is aligned to its size, so that a row of a set array in
// shared memory is one vector access.  A set in registers is only ever indexed by a word number known at compile time,
// or through compares on the agent (word_of, add_bit, drop_bit): a subscript known only at run time would put the set in
// local memory.
template <int W>
struct __align__(4 * W) Bits { uint32_t w[W]; };
template <int NC> using AgentSet = Bits<(NC > 64) ? 4 : 2>;

// agent i falls in word k of a W-word set (the last word takes every i >= 32 * (W - 1))
template <int W>
__device__ __forceinline__ bool in_word(int i, int k) { return (k == 0 || i >= 32 * k) && (k == W - 1 || i < 32 * k + 32); }
template <int W>
__device__ __forceinline__ uint32_t word_of(const Bits<W>& m, int i)   // the word that holds agent i
{
    uint32_t r = m.w[W - 1];
#pragma unroll
    for (int k = W - 2; k >= 0; --k) r = i < 32 * k + 32 ? m.w[k] : r;
    return r;
}
template <int W>
__device__ __forceinline__ bool bit_of(const Bits<W>& m, int i) { return (word_of(m, i) >> (i & 31)) & 1u; }
template <int W>
__device__ __forceinline__ void add_bit(Bits<W>& m, int i)
{
#pragma unroll
    for (int k = 0; k < W; ++k)
        if (in_word<W>(i, k)) m.w[k] |= 1u << (i & 31);
}
template <int W>
__device__ __forceinline__ void drop_bit(Bits<W>& m, int i)
{
#pragma unroll
    for (int k = 0; k < W; ++k)
        if (in_word<W>(i, k)) m.w[k] &= ~(1u << (i & 31));
}
// atomically adds agent `bit` to row r of a set array in shared memory (the word address: a compare for two words, a
// shift for four -- what ptxas turns into the fewer instructions at each width)
template <int W>
__device__ __forceinline__ void or_bit(Bits<W>* row, int r, int bit)
{
    atomicOr(W == 2 ? (bit < 32 ? &row[r].w[0] : &row[r].w[1]) : &row[r].w[bit >> 5], 1u << (bit & 31));
}
// the ballot of slot s (agents s*G .. s*G + G - 1) into a set that starts out empty: the first slot of a word assigns it
template <int G, int W>
__device__ __forceinline__ void put_slot(Bits<W>& m, int s, unsigned bm)
{
    const int k = (s * G) >> 5, sh = (s * G) & 31;
    m.w[k] = (sh ? m.w[k] : 0u) | (bm << sh);
}
template <int W>
__device__ __forceinline__ bool set_nonzero(const Bits<W>& m)
{
    uint32_t r = 0u;
#pragma unroll
    for (int k = 0; k < W; ++k) r |= m.w[k];
    return r != 0u;
}
template <int W>
__device__ __forceinline__ int set_count(const Bits<W>& m)
{
    int r = 0;
#pragma unroll
    for (int k = 0; k < W; ++k) r += __popc(m.w[k]);
    return r;
}
template <int W>
__device__ __forceinline__ int highest_of(const Bits<W>& m)   // the highest agent of the set, -1 if it is empty
{
    int r = -1;
#pragma unroll
    for (int k = W - 1; k >= 0; --k)
        if (r < 0 && m.w[k]) r = k * 32 + 31 - __clz((int)m.w[k]);
    return r;
}

// ------------------------------------------------------------------------------------------
// shared-memory layout of one environment
// ------------------------------------------------------------------------------------------
template <int NC>
struct Lay {
    static constexpr int POS = 0;                 // float2 [NC]  centre
    static constexpr int VEL = POS + 8 * NC;      // float2 [NC]  linear velocity
    static constexpr int FAT = VEL + 8 * NC;      // float4 [NC]  fat AABB lo.xy hi.xy
    static constexpr int ROWB = sizeof(AgentSet<NC>);   // bytes of one agent-set row
    static constexpr int ADJ = FAT + 16 * NC;     // set    [NC]  contact adjacency row (agents 0-31, 32-63, ...)
    // One agent-set row per agent of scratch, used by phases that never overlap in time:
    //   phase 1b  float2 [NC]  far end of an attacker's ray (TDM)
    //   phase 8   u32    [NC]  min sleep time of the island seeded here            (first half)
    //   phase 2a/10  set [NC]  new-pair row being assembled (re-zeroed on entry)
    //   phase 12-13  float [NC]  body angle for the TDM observation pass           (second half)
    static constexpr int NEW = ADJ + ROWB * NC;
    static constexpr int ISLMIN = NEW;
    static constexpr int ANG = NEW + 4 * NC;
    static constexpr int TGT = NEW + ROWB * NC;   // float2 [NC]  the agent's target (Flock), staged with the state
    static constexpr int TMASK = TGT + 8 * NC;    // u32    [NC]  staged touching contacts (index < 32) of a body
    static constexpr int LABEL = TMASK + 4 * NC;  // u32    [NC]  island seed (highest body index of the island)
    static constexpr int STACK = LABEL + 4 * NC;  // u8     [NC]  DFS stack (intrusive next-pointers on the common path)
    static constexpr int COMP = STACK + NC;       // u8     [NC]  seed body of the k-th island that has contacts
    static constexpr int SOLVED = COMP + NC;      // u8     [NC]  position solver converged for the island seeded here
    // dense piles only (more touching contacts than lanes, dense_* below):
    static constexpr int LASTLVL = SOLVED + NC, ISLACT = LASTLVL + NC, ISLBAD = ISLACT + NC;
    static constexpr int HEAD = ISLBAD + NC;      // u8     [NC]  newest touching contact of a body
    // 4 x u32; word 0, phases 5-7 of macm_kernels_huge.cu: contacts of a dense pile in the global-memory stage (0: the
    // env is in the shared-memory stage), from the velocity to the position part
    static constexpr int MISC = (HEAD + NC + 15) / 16 * 16;
    static constexpr int FIXED = MISC + 16;
    // per touching contact (capacity TC, a multiple of 16):
    //   float2 normal ; float2 impulses ; u32 edge word ; u16 slot ; u16 ord|lvl<<8    = 24 bytes
    __host__ __device__ static constexpr int bytes(int TC) { return (FIXED + 24 * TC + 15) / 16 * 16; }
};

// edge word of a touching contact: a | b<<B | next-of-a<<2B | next-of-b<<(2B+8) | taken<<(2B+16), B = 6 bits of body
// index for envs of up to 64 agents (the constants every shape had before 128-agent envs existed), 7 beyond
#define EW_NONE 255
template <int NC>
struct EW {
    static constexpr int B = NC > 64 ? 7 : 6;
    static constexpr uint32_t ID = (1u << B) - 1u, AB = (1u << (2 * B)) - 1u, TAKEN = 1u << (2 * B + 16);
    static constexpr int SH_B = B, SH_NA = 2 * B, SH_NB = 2 * B + 8;
    __device__ static int a(uint32_t w) { return (int)(w & ID); }
    __device__ static int b(uint32_t w) { return (int)((w >> SH_B) & ID); }
    __device__ static int na(uint32_t w) { return (int)((w >> SH_NA) & 255u); }
    __device__ static int nb(uint32_t w) { return (int)((w >> SH_NB) & 255u); }
};

template <int NC>
struct EnvS {
    unsigned char* base;
    int TC;
    __device__ float2* pos() const { return (float2*)(base + Lay<NC>::POS); }
    __device__ float2* vel() const { return (float2*)(base + Lay<NC>::VEL); }
    __device__ float4* fat() const { return (float4*)(base + Lay<NC>::FAT); }
    __device__ AgentSet<NC>* adj() const { return (AgentSet<NC>*)(base + Lay<NC>::ADJ); }
    __device__ AgentSet<NC>* nw() const { return (AgentSet<NC>*)(base + Lay<NC>::NEW); }
    __device__ uint32_t* isl_min() const { return (uint32_t*)(base + Lay<NC>::ISLMIN); }
    __device__ float* ang() const { return (float*)(base + Lay<NC>::ANG); }
    __device__ float2* tgt() const { return (float2*)(base + Lay<NC>::TGT); }
    __device__ uint32_t* tmask() const { return (uint32_t*)(base + Lay<NC>::TMASK); }
    __device__ uint32_t* label() const { return (uint32_t*)(base + Lay<NC>::LABEL); }
    __device__ uint8_t* stack() const { return base + Lay<NC>::STACK; }
    __device__ uint8_t* comp() const { return base + Lay<NC>::COMP; }
    __device__ uint8_t* solved() const { return base + Lay<NC>::SOLVED; }
    __device__ uint8_t* lastlvl() const { return base + Lay<NC>::LASTLVL; }
    __device__ uint8_t* isl_act() const { return base + Lay<NC>::ISLACT; }
    __device__ uint8_t* isl_bad() const { return base + Lay<NC>::ISLBAD; }
    __device__ uint8_t* head() const { return base + Lay<NC>::HEAD; }
    __device__ uint32_t* misc() const { return (uint32_t*)(base + Lay<NC>::MISC); }
    __device__ float2* t_n() const { return (float2*)(base + Lay<NC>::FIXED); }
    __device__ float2* t_imp() const { return t_n() + TC; }
    __device__ uint32_t* t_ew() const { return (uint32_t*)(t_n() + 2 * TC); }
    __device__ uint16_t* t_slot() const { return (uint16_t*)(t_ew() + TC); }
    __device__ uint16_t* ordlvl() const { return t_slot() + TC; }
};

// ------------------------------------------------------------------------------------------
// group-of-G-lanes primitives
// ------------------------------------------------------------------------------------------
template <int G>
struct Grp {
    unsigned mask;
    int shift, gl;
    __device__ Grp()
    {
        const int lane = threadIdx.x & 31;
        gl = lane % G;
        shift = lane - gl;
        mask = (G == 32) ? 0xffffffffu : (((1u << (G & 31)) - 1u) << shift);
    }
    __device__ unsigned ballot(bool p) const { return (__ballot_sync(mask, p) & mask) >> shift; }
    __device__ void sync() const { __syncwarp(mask); }
    __device__ unsigned below() const { return (1u << gl) - 1u; }
    __device__ unsigned reduce_min(unsigned v) const { return __reduce_min_sync(mask, v); }
    __device__ int shfl(int v, int src) const { return __shfl_sync(mask, v, shift + src); }
    // inclusive prefix sum over the group lanes
    __device__ int scan_incl(int v) const
    {
#pragma unroll
        for (int d = 1; d < G; d <<= 1) {
            int o = __shfl_up_sync(mask, v, d, G);
            if (gl >= d) v += o;
        }
        return v;
    }
};

// Packed fp32x2 arithmetic of sm_100 (FADD2 / FMUL2): two IEEE round-to-nearest operations per
// instruction, bit-identical to the scalar ones.  (A packed multiply feeding a packed add would be
// contracted into FFMA2 by ptxas even with .rn, so sums of products are finished with scalar adds.)
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) { f32x2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }

// pull `bytes` starting at p towards L2, one 128-byte line per lane of the group
template <int G>
__device__ __forceinline__ void prefetch_l2(int gl, const void* p, int bytes)
{
    for (int off = gl * 128; off < bytes; off += G * 128)
        asm volatile("prefetch.global.L2 [%0];" ::"l"((const char*)p + off));
}

// b2TestOverlap(b2AABB, b2AABB): d1 = b.lo - a.hi, d2 = a.lo - b.hi; overlap iff no component > 0.
// With IEEE gradual underflow (no -ftz) x - y > 0 <=> x > y, so the subtractions are not needed.
__device__ __forceinline__ bool aabb_overlap(const float4 a, const float4 b)
{
    return !(b.x > a.z || b.y > a.w || a.x > b.z || a.y > b.w);
}

__device__ __forceinline__ float b2min(float a, float b) { return a < b ? a : b; }
__device__ __forceinline__ float b2max(float a, float b) { return a > b ? a : b; }
__device__ __forceinline__ float b2clamp(float a, float lo, float hi) { return b2max(lo, b2min(a, hi)); }

// b2Vec2::Normalize (unchanged when shorter than b2_epsilon)
__device__ __forceinline__ void b2normalize(float& x, float& y)
{
    float len = sqrtf(x * x + y * y);
    if (len < B2_EPSILON) return;
    float inv = 1.0f / len;
    x *= inv;
    y *= inv;
}

// sqrt for OUTPUTS only (observation distances, the linear reward): the reference computes them in
// float64, the tests hold these floats to 1e-5 relative, and sqrt.approx is good to 1 ulp of fp32.
// Engine state never goes through it (b2normalize, the translation clamp and the ray cast keep IEEE sqrtf).
__device__ __forceinline__ float out_sqrtf(float x) { float r; asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

// Two fp32 observation values -> one word of two 16-bit ones (MACM_OBS_F16 / MACM_OBS_BF16), `lo` at the lower
// address; rounded to nearest even, with subnormals kept (no .ftz), as torch's .to(float16 / bfloat16) rounds.
// The PTX form puts its FIRST source in the upper half.
__device__ __forceinline__ uint32_t obs_pack2(float lo, float hi, bool bf16)
{
    uint32_t r;
    if (bf16) asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    else asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// one 4-value observation record at the element type of `Rec`: float4 (fp32) or uint2 (four 16-bit values)
template <typename Rec> __device__ __forceinline__ Rec obs_record(float4 v, bool bf16);
template <> __device__ __forceinline__ float4 obs_record<float4>(float4 v, bool) { return v; }
template <> __device__ __forceinline__ uint2 obs_record<uint2>(float4 v, bool bf16)
{
    return make_uint2(obs_pack2(v.x, v.y, bf16), obs_pack2(v.z, v.w, bf16));
}

// t - sign(t)*2*pi if |t| > pi else t (mvmnt.py:199), in fp32 for the observation outputs
__device__ __forceinline__ float wrap_pi_f(float t)
{
    const float PI_F = 3.14159265358979f, TWO_PI_F = 6.28318530717959f;
    if (fabsf(t) > PI_F) t = t - copysignf(TWO_PI_F, t);
    return t;
}

// atan2 for the observation outputs (fp32, reference: float64 np.arctan2): octant reduction +
// degree-15 odd minimax polynomial, max error 1.3e-7 rad over the reduced range (measured against
// float64 atan with the float32 evaluation order below); tests allow 3e-6.
__device__ __forceinline__ float fast_atan2f(float y, float x)
{
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const float a = mx > 0.0f ? __fdividef(mn, mx) : 0.0f;
    const float q = a * a;
    float r = -0.0040545230731368065f;
    r = fmaf(r, q, 0.02186279185116291f);
    r = fmaf(r, q, -0.0559120774269104f);
    r = fmaf(r, q, 0.09642177820205688f);
    r = fmaf(r, q, -0.13908621668815613f);
    r = fmaf(r, q, 0.19946564733982086f);
    r = fmaf(r, q, -0.33329859375953674f);
    r = fmaf(r, q, 0.9999993443489075f);
    r = r * a;
    if (ay > ax) r = 1.5707963267948966f - r;
    if (x < 0.0f) r = 3.14159265358979f - r;
    return copysignf(r, y);
}

__device__ __noinline__ void sincos_slow(float Af, double* s, double* c) { sincos((double)Af, s, c); }

// sin and cos of a float32 angle to ~1 ulp of float64.  A = k/128 + x with |x| <= 2^-8 (exact
// split, A is a float): table of sin/cos(k/128) (host-computed doubles) + degree-7/8 Taylor.
// Outside the table (|A| > 3.25, only reachable through load_state) falls back to sincos().
__device__ __forceinline__ void sincos_f32arg(const double2* __restrict__ tab, float Af, double& s, double& c)
{
    const float fk = rintf(fabsf(Af) * 128.0f);
    if (!(fk <= 416.0f)) { sincos_slow(Af, &s, &c); return; }
    const double2 sc = tab[(int)fk];
    const double x = fabs((double)Af) - (double)fk * 0.0078125;
    const double x2 = x * x;
    // sin x = x + x^3 (-1/6 + x^2 (1/120 - x^2/5040)) ; cos x - 1 = x^2 (-1/2 + x^2 (1/24 + x^2 (-1/720 + x^2/40320)))
    const double ps = fma(x2, fma(x2, -1.984126984126984e-04, 8.333333333333333e-03), -1.6666666666666666e-01);
    const double sl = fma(x * x2, ps, x);
    const double dc = x2 * fma(x2, fma(x2, fma(x2, 2.48015873015873e-05, -1.388888888888889e-03), 4.1666666666666664e-02), -0.5);
    const double sa = sc.x + fma(sc.y, sl, sc.x * dc);
    c = sc.y + fma(sc.y, dc, -(sc.x * sl));
    s = (Af < 0.0f) ? -sa : sa;
}

// One velocity-constraint pass of one contact (b2ContactSolver::SolveVelocityConstraints,
// pointCount == 1, invI = 0): tangent (friction) first, then normal.
__device__ __forceinline__ void solve_velocity(float nx, float ny, float friction, float mass_n, float mass_t,
                                               float inv_mass, float& nI, float& tI, float2& va, float2& vb)
{
    const float tx = ny, ty = -nx;  // b2Cross(normal, 1.0f)
    {
        float dvx = vb.x - va.x, dvy = vb.y - va.y;
        float vt = dvx * tx + dvy * ty;
        float lambda = mass_t * (-vt);
        float maxf = friction * nI;
        float ni = b2clamp(tI + lambda, -maxf, maxf);
        lambda = ni - tI;
        tI = ni;
        float Px = lambda * tx, Py = lambda * ty;
        va.x -= inv_mass * Px; va.y -= inv_mass * Py;
        vb.x += inv_mass * Px; vb.y += inv_mass * Py;
    }
    {
        float dvx = vb.x - va.x, dvy = vb.y - va.y;
        float vn = dvx * nx + dvy * ny;
        float lambda = -mass_n * vn;
        float ni = b2max(nI + lambda, 0.0f);
        lambda = ni - nI;
        nI = ni;
        float Px = lambda * nx, Py = lambda * ny;
        va.x -= inv_mass * Px; va.y -= inv_mass * Py;
        vb.x += inv_mass * Px; vb.y += inv_mass * Py;
    }
}

// b2ContactSolver::WarmStart of one contact
__device__ __forceinline__ void warm_start(float nx, float ny, float nI, float tI, float inv_mass, float2& va, float2& vb)
{
    const float tx = ny, ty = -nx;
    const float Px = nI * nx + tI * tx, Py = nI * ny + tI * ty;
    va.x -= inv_mass * Px; va.y -= inv_mass * Py;
    vb.x += inv_mass * Px; vb.y += inv_mass * Py;
}

// One position-constraint pass of one contact (b2ContactSolver::SolvePositionConstraints +
// b2PositionSolverManifold::Initialize, e_circles).  Returns the separation it saw.
__device__ __forceinline__ float solve_position(float radius, float k_sum, float inv_mass, float2& ca, float2& cb)
{
    float nx = cb.x - ca.x, ny = cb.y - ca.y;
    const float dx = nx, dy = ny;
    b2normalize(nx, ny);
    float sep = (dx * nx + dy * ny) - radius - radius;
    float C = b2clamp(B2_BAUMGARTE * (sep + B2_LINEAR_SLOP), -B2_MAX_LINEAR_CORRECTION, 0.0f);
    float imp = k_sum > 0.0f ? -C / k_sum : 0.0f;
    float Px = imp * nx, Py = imp * ny;
    ca.x -= inv_mass * Px; ca.y -= inv_mass * Py;
    cb.x += inv_mass * Px; cb.y += inv_mass * Py;
    return sep;
}

// ------------------------------------------------------------------------------------------
// b2ContactManager::FindNewContacts for one environment (group-cooperative).
//   moved: set of proxies in the broadphase move buffer.
//   Every other proxy whose fat AABB overlaps a moved one forms a pair; pairs are sorted
//   lexicographically, de-duplicated, and those without a contact yet are created in that
//   order (lower index = fixtureA).  Here: row i of a bit matrix holds the partners j > i;
//   emitting rows in index order and bits in ascending order IS the sorted order.
// Appends to the HBM contact list at `cnt`; returns the new count (uniform over the group).
// ------------------------------------------------------------------------------------------
template <int G, int APL>
__device__ int find_new_contacts(const Grp<G>& g, const EnvS<G * APL>& S, const SimConst& P, const AgentSet<G * APL>& moved,
                                 const AgentSet<G * APL>& alive, int cnt, uint32_t* c_ab, float2* c_imp, bool& overflow)
{
    typedef AgentSet<G * APL> Set;
    constexpr int W = sizeof(Set) / 4, NW = (G * APL + 31) / 32;   // words of a set, words that can hold an agent
    const float4* fat = S.fat();
    Set* adj = S.adj();
    Set* nw = S.nw();

    Set hit[APL];
    float4 own[APL];
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        hit[s] = Set{};
        own[s] = fat[i];
        // dead / padding agents have no proxy: park their box where nothing overlaps it
        if (!bit_of(alive, i)) own[s] = make_float4(3.0e38f, 3.0e38f, -3.0e38f, -3.0e38f);
        nw[i] = Set{};
    }
    g.sync();
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        for (unsigned mm = moved.w[w]; mm; mm &= mm - 1) {
            const int m = w * 32 + __ffs((int)mm) - 1;
            const float4 mb = fat[m];
            const unsigned bit = 1u << (m & 31);
#pragma unroll
            for (int s = 0; s < APL; ++s) {
                const bool h = (g.gl + s * G != m) && aabb_overlap(mb, own[s]);
                hit[s].w[w] |= h ? bit : 0u;
            }
        }
    }
    // pair (m, i) with m < i belongs to row m: the owner of m finds it itself iff i moved too;
    // otherwise the owner of i posts it
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        if (!bit_of(moved, i)) {
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                unsigned lo = hit[s].w[w];
                if (in_word<W>(i, w)) lo &= (1u << (i & 31)) - 1u;   // partners m < i only
                if (w > 0 && i < 32 * w) lo = 0u;
                for (; lo; lo &= lo - 1) or_bit(nw, w * 32 + __ffs((int)lo) - 1, i);
            }
        }
    }
    g.sync();
    Set fresh[APL];
    bool any = false;
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        const Set posted = nw[i], have = adj[i];
        fresh[s] = Set{};
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            unsigned row = hit[s].w[w];
            if (in_word<W>(i, w)) row &= ~((2u << (i & 31)) - 1u);   // keep partners j > i only
            if (w < W - 1 && i >= 32 * w + 32) row = 0u;
            fresh[s].w[w] = (row | posted.w[w]) & ~have.w[w];
        }
        any |= set_nonzero(fresh[s]);
    }
    if (!g.ballot(any)) return cnt;
    int base = cnt;
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        const int c = set_count(fresh[s]);
        const int incl = g.scan_incl(c);
        const int total = g.shfl(incl, G - 1);
        int pos = base + incl - c;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            for (unsigned f = fresh[s].w[w]; f; f &= f - 1) {
                const int j = w * 32 + __ffs((int)f) - 1;
                if (pos < P.C) {
                    c_ab[pos] = (uint32_t)i | ((uint32_t)j << 8);
                    c_imp[pos] = make_float2(0.0f, 0.0f);
                    or_bit(adj, i, j);
                    or_bit(adj, j, i);
                } else {
                    overflow = true;
                }
                ++pos;
            }
        }
        base += total;
    }
    g.sync();
    return base < P.C ? base : P.C;
}

// ------------------------------------------------------------------------------------------
// Nearest other agent for the two agents of a lane (N in 33..64; agents gl and gl + 32).
//
// The select/compare pipe is the scarce one on this path (16 lanes per sub-partition against 32 for
// the FMA pipes), so the search spends its work on the FMA side: squared distances in packed fp32x2
// (lo half = the lane's first agent, hi half = its second) and, per block of four candidates, one
// 3-input min + min + compare + select per agent -- the running minimum and the BLOCK it came from.
// The index inside the block is recovered afterwards by recomputing four distances.
//
// Positions are staged as P4[j] = (x_j, x_{j+32}, y_j, y_{j+32}), j = 0..31, twice in a row, so that
//   * the lane's own half (agents of the same 32-block) is read at P4[gl + r], r = 1..31: every
//     other agent of the block exactly once, never itself, no index arithmetic, no self test;
//   * the other half is read at P4[j], j = 0..31 (broadcast), against the lane's agents swapped.
// The reference keeps the lowest index among equal minima (strict '<' in ascending order,
// mvmnt.py:194).  The broadcast half is visited in ascending order, so there the first block wins
// and the lowest index inside it is taken; the rotated half is not, so an exact tie between a
// block's minimum and the running minimum raises a flag and that agent is searched again, exactly, by
// the whole group (nn_rescan; about 3 % of the warps have such an agent in a step).
// ------------------------------------------------------------------------------------------
// Exact nearest other agent of ONE agent (position o, index self), by the whole group: lane j looks at
// candidates j and j + 32, the minimum goes through a warp reduction on the bit patterns (squared
// distances are non-negative, so unsigned order is float order) and the lowest index holding it wins.
template <int G>
__device__ __noinline__ float2 nn_rescan(const Grp<G>& g, const float2* pos, float2 o, int self)
{
    const float2 qa = pos[g.gl], qb = pos[g.gl + 32];
    const float ax = qa.x - o.x, ay = qa.y - o.y, bx = qb.x - o.x, by = qb.y - o.y;
    unsigned da = __float_as_uint(ax * ax + ay * ay), db = __float_as_uint(bx * bx + by * by);
    if (g.gl == self) da = 0xffffffffu;
    if (g.gl + 32 == self) db = 0xffffffffu;
    const unsigned m = __reduce_min_sync(g.mask, min(da, db));
    const unsigned la = g.ballot(da == m), lb = g.ballot(db == m);
    const int idx = la ? (__ffs((int)la) - 1) : (32 + __ffs((int)lb) - 1);
    return make_float2(__uint_as_float(m), __int_as_float(idx));
}

#define NN_D2(q, OX, OY, dl, dh)                                                             \
    {                                                                                        \
        const f32x2 dx_ = sub2(pack2((q).x, (q).y), OX), dy_ = sub2(pack2((q).z, (q).w), OY); \
        float xl_, xh_, yl_, yh_;                                                            \
        unpack2(mul2(dx_, dx_), xl_, xh_);                                                   \
        unpack2(mul2(dy_, dy_), yl_, yh_);                                                   \
        dl = __fadd_rn(xl_, yl_); dh = __fadd_rn(xh_, yh_);   /* b2DistanceSquared, no FMA */ \
    }

template <int G>
__device__ __forceinline__ void nn_search_64(const Grp<G>& g, const EnvS<2 * G>& S, float2 o0, float2 o1,
                                             float& best0, int& bi0, float& best1, int& bi1)
{
    static_assert(G == 32, "two agents per lane means 32 lanes per env");
    const float2* pos = S.pos();
    float4* P4 = reinterpret_cast<float4*>(S.fat());   // the fat AABBs are dead by now
    g.sync();
    P4[g.gl] = P4[g.gl + 32] = make_float4(o0.x, o1.x, o0.y, o1.y);
    g.sync();
    const float BIG = 3.4028234664e38f;   // every real squared distance is below it; padding agents give +inf
    const f32x2 ox = pack2(o0.x, o1.x), oy = pack2(o0.y, o1.y);      // own half: lo = agent gl, hi = agent gl + 32
    const f32x2 oxs = pack2(o1.x, o0.x), oys = pack2(o1.y, o0.y);    // other half: lo = agent gl + 32 against A_j, hi = agent gl against B_j
    float bo0 = BIG, bo1 = BIG, bc0 = BIG, bc1 = BIG;   // running minima: own half (agent 0, agent 1), other half
    int ko0 = 0, ko1 = 0, kc0 = 0, kc1 = 0;              // first candidate of the block of the minimum
    // smallest |block minimum - running minimum| seen: exactly 0 <=> an exact draw (the subtraction goes
    // to the FMA pipe, the |.| min is one op on the other)
    float tz0 = BIG, tz1 = BIG;
    const float4* own = P4 + g.gl + 1;
    // (the loop counter doubles as the block id: one add and one compare per block)
#pragma unroll 1
    for (int b = 0; b < 28; b += 4) {
        float dl[4], dh[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { const float4 q = own[b + k]; NN_D2(q, ox, oy, dl[k], dh[k]); }
        const float ml = fminf(fminf(fminf(dl[0], dl[1]), dl[2]), dl[3]), mh = fminf(fminf(fminf(dh[0], dh[1]), dh[2]), dh[3]);
        tz0 = fminf(tz0, fabsf(ml - bo0)); tz1 = fminf(tz1, fabsf(mh - bo1));
        const bool pl = ml < bo0, ph = mh < bo1;
        bo0 = fminf(bo0, ml); bo1 = fminf(bo1, mh);
        ko0 = pl ? b : ko0; ko1 = ph ? b : ko1;
    }
    {   // r = 29, 30, 31
        float dl[3], dh[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) { const float4 q = own[28 + k]; NN_D2(q, ox, oy, dl[k], dh[k]); }
        const float ml = fminf(fminf(dl[0], dl[1]), dl[2]), mh = fminf(fminf(dh[0], dh[1]), dh[2]);
        tz0 = fminf(tz0, fabsf(ml - bo0)); tz1 = fminf(tz1, fabsf(mh - bo1));
        const bool pl = ml < bo0, ph = mh < bo1;
        bo0 = fminf(bo0, ml); bo1 = fminf(bo1, mh);
        ko0 = pl ? 28 : ko0; ko1 = ph ? 28 : ko1;
    }
    const bool tie0 = tz0 == 0.0f, tie1 = tz1 == 0.0f;
#pragma unroll 1
    for (int b = 0; b < 32; b += 4) {
        float dl[4], dh[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { const float4 q = P4[b + k]; NN_D2(q, oxs, oys, dl[k], dh[k]); }
        // lo: agent gl + 32 against A_j ; hi: agent gl against B_j
        const float ml = fminf(fminf(fminf(dl[0], dl[1]), dl[2]), dl[3]), mh = fminf(fminf(fminf(dh[0], dh[1]), dh[2]), dh[3]);
        const bool pl = ml < bc1, ph = mh < bc0;
        bc1 = fminf(bc1, ml); bc0 = fminf(bc0, mh);
        kc1 = pl ? b : kc1; kc0 = ph ? b : kc0;
    }
    // agent gl: its own half holds the lower indices, so it wins an exact draw; agent gl + 32: the other half does
    const bool own0 = bo0 <= bc0, own1 = bo1 < bc1;
    best0 = own0 ? bo0 : bc0;
    best1 = own1 ? bo1 : bc1;
    bi0 = 64; bi1 = 64;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int r0 = 1 + ko0 + k, r1 = 1 + ko1 + k;
        const int c0 = own0 ? ((g.gl + r0) & 31) : (32 + kc0 + k);
        const int c1 = own1 ? (32 + ((g.gl + r1) & 31)) : (kc1 + k);
        const bool in0 = !own0 || r0 < 32, in1 = !own1 || r1 < 32;
        const float2 q0 = pos[c0], q1 = pos[c1];
        const float ax = q0.x - o0.x, ay = q0.y - o0.y, bx = q1.x - o1.x, by = q1.y - o1.y;
        const float d0 = ax * ax + ay * ay, d1 = bx * bx + by * by;
        if (in0 && d0 == best0) bi0 = min(bi0, c0);
        if (in1 && d1 == best1) bi1 = min(bi1, c1);
    }
    // an exact draw in the rotated half (about one agent in 4,000: two of its 63 squared distances collide):
    // that agent is searched again, exactly, by the whole group
    {
        unsigned n0 = g.ballot((own0 && tie0) || bi0 == 64), n1 = g.ballot((own1 && tie1) || bi1 == 64);
        for (; n0; n0 &= n0 - 1) {
            const int src = __ffs((int)n0) - 1;
            const float2 oo = make_float2(__shfl_sync(g.mask, o0.x, src), __shfl_sync(g.mask, o0.y, src));
            const float2 r = nn_rescan<G>(g, pos, oo, src);
            if (g.gl == src) { best0 = r.x; bi0 = __float_as_int(r.y); }
        }
        for (; n1; n1 &= n1 - 1) {
            const int src = __ffs((int)n1) - 1;
            const float2 oo = make_float2(__shfl_sync(g.mask, o1.x, src), __shfl_sync(g.mask, o1.y, src));
            const float2 r = nn_rescan<G>(g, pos, oo, src + 32);
            if (g.gl == src) { best1 = r.x; bi1 = __float_as_int(r.y); }
        }
    }
}

// Nearest other agent for the FOUR agents of a lane (N in 65..128; agents gl, gl + 32, gl + 64, gl + 96).
// Every candidate is broadcast in ascending index order, so strict '<' between blocks of four and the lowest index
// inside the winning block IS the reference's tie-break (mvmnt.py:194) -- no re-scan needed; the price is an explicit
// self test, paid only by the slot whose own 32-block is being visited (the loop is unrolled over the four blocks).
// Squared distances in packed fp32x2 for the agent pairs (0, 1) and (2, 3): positions are staged as
// (x, x, y, y), so the two operand pairs of a candidate come out of one 16-byte load.
template <int G>
__device__ __forceinline__ void nn_search_128(const Grp<G>& g, const EnvS<4 * G>& S, const float2 (&o)[4], float (&best)[4],
                                              int (&bi)[4])
{
    static_assert(G == 32, "four agents per lane means 32 lanes per env");
    const float2* pos = S.pos();
    float4* P4 = reinterpret_cast<float4*>(S.fat());   // the fat AABBs are dead by now
    g.sync();
#pragma unroll
    for (int s = 0; s < 4; ++s) P4[g.gl + 32 * s] = make_float4(o[s].x, o[s].x, o[s].y, o[s].y);
    g.sync();
    const float BIG = 3.4028234664e38f;   // every real squared distance is below it; padding agents give +inf
    const f32x2 ox01 = pack2(o[0].x, o[1].x), oy01 = pack2(o[0].y, o[1].y);
    const f32x2 ox23 = pack2(o[2].x, o[3].x), oy23 = pack2(o[2].y, o[3].y);
    float bm[4] = {BIG, BIG, BIG, BIG};   // running minimum per agent
    int kb[4] = {0, 0, 0, 0};             // first candidate of the block of four it came from
#pragma unroll
    for (int blk = 0; blk < 4; ++blk) {   // the 32-block that holds this lane's agent `blk`
#pragma unroll 1
        for (int b = 32 * blk; b < 32 * blk + 32; b += 4) {
            float d[4][4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float4 q = P4[b + k];
                const f32x2 qx = pack2(q.x, q.y), qy = pack2(q.z, q.w);
                const f32x2 dx01 = sub2(qx, ox01), dy01 = sub2(qy, oy01), dx23 = sub2(qx, ox23), dy23 = sub2(qy, oy23);
                float xl, xh, yl, yh;
                unpack2(mul2(dx01, dx01), xl, xh); unpack2(mul2(dy01, dy01), yl, yh);
                d[k][0] = __fadd_rn(xl, yl); d[k][1] = __fadd_rn(xh, yh);   // b2DistanceSquared, no FMA
                unpack2(mul2(dx23, dx23), xl, xh); unpack2(mul2(dy23, dy23), yl, yh);
                d[k][2] = __fadd_rn(xl, yl); d[k][3] = __fadd_rn(xh, yh);
                if (b + k - 32 * blk == g.gl) d[k][blk] = BIG;              // an agent is not its own neighbour
            }
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const float m = fminf(fminf(fminf(d[0][s], d[1][s]), d[2][s]), d[3][s]);
                const bool p = m < bm[s];
                bm[s] = fminf(bm[s], m);
                kb[s] = p ? b : kb[s];
            }
        }
    }
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        best[s] = bm[s];
        bi[s] = 128;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = kb[s] + k;
            const float2 q = pos[c];
            const float ax = q.x - o[s].x, ay = q.y - o[s].y;
            const float dd = ax * ax + ay * ay;
            if (c != g.gl + 32 * s && dd == bm[s]) bi[s] = min(bi[s], c);
        }
    }
}

// ------------------------------------------------------------------------------------------
// observation pass for the agents a lane owns (Flock.get_obs, mvmnt.py:181-222)
// ------------------------------------------------------------------------------------------
// cartesian variant of the observation record (coord == "cartesian", mvmnt.py:202-203,215-216); cold.
// 24 bytes per agent in fp32, 12 (three words) at a 16-bit obs_dtype.
__device__ __noinline__ void store_cartesian(float* obs, size_t gi, float nn_d, float nn_t, float tg_r, float tg_t,
                                             int dtype)
{
    float sn, cn, st, ct;
    sincosf(nn_t, &sn, &cn);
    sincosf(tg_t, &st, &ct);
    if (dtype == MACM_OBS_F32) {
        float2* ob = reinterpret_cast<float2*>(obs) + gi * 3;
        ob[0] = make_float2(nn_d, cn);
        ob[1] = make_float2(sn, tg_r);
        ob[2] = make_float2(ct, st);
    } else {
        const bool bf16 = dtype == MACM_OBS_BF16;
        uint32_t* ob = reinterpret_cast<uint32_t*>(obs) + gi * 3;
        ob[0] = obs_pack2(nn_d, cn, bf16);
        ob[1] = obs_pack2(sn, tg_r, bf16);
        ob[2] = obs_pack2(ct, st, bf16);
    }
}

// Destinations: (ob1, nn1) and (ob2, nn2), each pointer may be null (a rollout writes a step's observation to
// the caller's per-step arrays and, on its last step, to the sim's bound buffers as well).  tgo, when not null,
// receives every agent's target node (r, theta), indexed by agent -- what the flock actor of bots.py steers by.
template <int G, int APL>
__device__ void flock_observe(const Grp<G>& g, const EnvS<G * APL>& S, const SimConst& P, int env, const float* ang,
                              float* ob1, int* nn1, float* ob2, int* nn2, float2* tgo = nullptr)
{
    const float2* pos = S.pos();
    const int N = P.N;
    float2 o[APL], tg[APL];
    float best[APL];
    int bi[APL];
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        o[s] = pos[i];
        best[s] = __int_as_float(0x7f800000);
        bi[s] = -1;
    }
    // nearest other agent: strict '<' over ascending j keeps the lowest index on ties (mvmnt.py:194).
    // Slot s only has to skip itself while j runs through its own 32-block.
    if constexpr (APL == 2) {
        nn_search_64<G>(g, S, o[0], o[APL - 1], best[0], bi[0], best[APL - 1], bi[APL - 1]);
    } else if constexpr (APL == 4) {
        nn_search_128<G>(g, S, o, best, bi);
    } else {
#pragma unroll
        for (int jb = 0; jb < G * APL; jb += G) {
            const int jend = (N - jb) < G ? (N - jb) : G;
#pragma unroll 4
            for (int jj = 0; jj < jend; ++jj) {
                const float2 q = pos[jb + jj];
                const bool notme = jj != g.gl;
#pragma unroll
                for (int s = 0; s < APL; ++s) {
                    const float dx = q.x - o[s].x, dy = q.y - o[s].y;
                    const float d2 = dx * dx + dy * dy;  // b2DistanceSquared, no FMA
                    const bool take = (s * G == jb) ? ((d2 < best[s]) && notme) : (d2 < best[s]);
                    best[s] = take ? d2 : best[s];
                    bi[s] = take ? (jb + jj) : bi[s];
                }
            }
        }
    }
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        if (i >= N) continue;
        tg[s] = S.tgt()[i];
        const size_t gi = (size_t)env * N + i;
        float nn_d = __int_as_float(0x7f800000), nn_t = 0.0f;
        if (bi[s] >= 0) {
            const float2 q = pos[bi[s]];
            nn_d = out_sqrtf(best[s]);
            nn_t = wrap_pi_f(fast_atan2f(q.y - o[s].y, q.x - o[s].x) - ang[s]);
        }
        const float tdx = tg[s].x - o[s].x, tdy = tg[s].y - o[s].y;
        const float tg_r = out_sqrtf(tdx * tdx + tdy * tdy);
        const float tg_t = wrap_pi_f(fast_atan2f(tdy, tdx) - ang[s]);
        if (tgo) tgo[i] = make_float2(tg_r, tg_t);
        if (nn1) nn1[gi] = bi[s];
        if (nn2) nn2[gi] = bi[s];
        if (P.coord == MACM_COORD_POLAR) {
            const float4 o4 = make_float4(nn_d, nn_t, tg_r, tg_t);
            if (P.obs_dtype == MACM_OBS_F32) {
                if (ob1) reinterpret_cast<float4*>(ob1)[gi] = o4;
                if (ob2) reinterpret_cast<float4*>(ob2)[gi] = o4;
            } else {
                const uint2 w = obs_record<uint2>(o4, P.obs_dtype == MACM_OBS_BF16);
                if (ob1) reinterpret_cast<uint2*>(ob1)[gi] = w;
                if (ob2) reinterpret_cast<uint2*>(ob2)[gi] = w;
            }
        } else {
            if (ob1) store_cartesian(ob1, gi, nn_d, nn_t, tg_r, tg_t, P.obs_dtype);
            if (ob2) store_cartesian(ob2, gi, nn_d, nn_t, tg_r, tg_t, P.obs_dtype);
        }
    }
}

// The N x N records of one env, walked in MEMORY order, G at a time (record r = i * N + j -> lane r % G): every store
// of the group is one contiguous run of records whatever N is, and no lane idles on a ragged row end (N = 45 on 32
// lanes: 64 rounds instead of 90).  i and j advance without a division.  Rec is the record as stored: float4, or
// uint2 for four 16-bit values -- chosen once per call, so that the fp32 loop carries no conversion.
template <int G, typename Rec>
__device__ __forceinline__ void tdm_rows(const Grp<G>& g, const float4* hdr, int N, Rec* out, Rec* out2, bool bf16)
{
    const int total = N * N;
    int i = g.gl / N, j = g.gl - i * N;          // G may exceed N (small teams on a wide group)
    const int di = G / N, dj = G - di * N;       // one round further: G records
#pragma unroll 1
    for (int r = g.gl; r < total; r += G) {
        const float4 h = hdr[i];   // observer: x, y, heading, team (-1: dead, observes nothing)
        const float4 q = hdr[j];   // observed
        const float dx = q.x - h.x, dy = q.y - h.y;
        const bool entry = h.w >= 0.0f && q.w >= 0.0f && j != i;
        float4 v;
        v.x = entry ? out_sqrtf(dx * dx + dy * dy) : 0.0f;
        v.y = entry ? wrap_pi_f(fast_atan2f(dy, dx) - h.z) : 0.0f;
        v.z = entry ? wrap_pi_f(q.z - h.z) : 0.0f;
        v.w = entry ? ((q.w == h.w) ? 1.0f : 0.0f) : -1.0f;
        const Rec rec = obs_record<Rec>(v, bf16);
        if (out) out[r] = rec;
        if (out2) out2[r] = rec;
        j += dj; i += di;
        if (j >= N) { j -= N; ++i; }
    }
}

// TDM.get_obs (combat.py:206-227): for every alive agent i, every other alive agent j:
// [r, theta, phi] and the ally flag.  Row i of the [N,N,4] output is written by the whole group
// (lane <-> j) so that the record stores of a row are contiguous.
// The pass is the bulk of a TDM step (N^2 records of 16 bytes: 70 % of its instructions), so the row loop is kept
// lean: one 16-byte header per agent (x, y, heading, team -- or -1 when it has no entry) staged where the fat AABBs
// lived (dead by now, as in nn_search_64), one broadcast load per row, no branch inside the row (a record without
// an entry is selected, not jumped around), row pointers advanced instead of recomputed.
template <int G, int APL>
__device__ void tdm_observe(const Grp<G>& g, const EnvS<G * APL>& S, const SimConst& P, int env,
                            const AgentSet<G * APL>& alive, float* ob1, float* ob2)
{
    const float2* pos = S.pos();
    const float* angs = S.ang();
    const int N = P.N;
    float4* hdr = S.fat();
    g.sync();
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int j = g.gl + s * G;
        const float2 q = pos[j];
        hdr[j] = make_float4(q.x, q.y, angs[j], (j < N && bit_of(alive, j)) ? (float)P.team[j] : -1.0f);
    }
    g.sync();
    const size_t first = (size_t)env * N * N;   // the env's first record
    if (P.obs_dtype == MACM_OBS_F32) {
        tdm_rows<G>(g, hdr, N, ob1 ? reinterpret_cast<float4*>(ob1) + first : nullptr,
                    ob2 ? reinterpret_cast<float4*>(ob2) + first : nullptr, false);
    } else {
        tdm_rows<G>(g, hdr, N, ob1 ? reinterpret_cast<uint2*>(ob1) + first : nullptr,
                    ob2 ? reinterpret_cast<uint2*>(ob2) + first : nullptr, P.obs_dtype == MACM_OBS_BF16);
    }
}

// ------------------------------------------------------------------------------------------
// Dense piles: environments with more touching contacts than lanes (tc > G).  One lane replays Box2D's depth-first
// island traversal over per-body edge lists (head-inserted in birth order, like b2ContactManager::AddPair builds them);
// every contact gets its position in the island order and a level = 1 + max(level of the previous contact of either
// body).  Contacts of one level share no body and run across lanes.  Rare, and kept out of line so that the common path
// stays small in the instruction cache.
//
// The solver is written once, on a STAGE: where the env's touching contacts live while they are ordered and solved.
//   SmemStage  the shared-memory stage that phase 2 fills (capacity TC <= 240): the next-links of a contact are bytes of
//              its edge word, order and level a u16 t | lvl<<8, head / lastlvl a byte per body.
//   GmemStage  the global-memory stage (macm_buffers.touch_scratch, max_touching > 240; only in the kernels of
//              macm_kernels_huge.cu): 16-bit links, order and levels.  It takes envs with more than TC touching contacts
//              -- overlapping spawn piles; bodies that do not overlap cannot touch more than ~3N others.  Without it such
//              an env is flagged MACM_ENV_TOUCH_OVERFLOW instead.
// A stage provides edge(t) -> w, a(w) / b(w), next(w, t, body) (the next edge at `body`), link(t, w, next-of-a,
// next-of-b), taken(w) / take(t, w), ord(k) -> (t, lvl) / set_ord(k, t, lvl), the arrays n, imp (normal and impulses of
// contact t) and slot (its HBM list index), head / lastlvl (per body), and NONE (end of an edge list).
// ------------------------------------------------------------------------------------------
template <int NC>
struct SmemStage {
    typedef EW<NC> E;
    static constexpr int NONE = EW_NONE;
    uint32_t* ew; uint16_t* ol; float2* n; float2* imp; uint16_t* slot; uint8_t* head; uint8_t* lastlvl;
    __device__ explicit SmemStage(const EnvS<NC>& S)
        : ew(S.t_ew()), ol(S.ordlvl()), n(S.t_n()), imp(S.t_imp()), slot(S.t_slot()), head(S.head()), lastlvl(S.lastlvl()) {}
    __device__ uint32_t edge(int t) const { return ew[t]; }
    __device__ static int a(uint32_t w) { return E::a(w); }
    __device__ static int b(uint32_t w) { return E::b(w); }
    __device__ int next(uint32_t w, int, int body) const { return a(w) == body ? E::na(w) : E::nb(w); }
    __device__ void link(int t, uint32_t w, int na, int nb) const { ew[t] = w | ((uint32_t)na << E::SH_NA) | ((uint32_t)nb << E::SH_NB); }
    __device__ static bool taken(uint32_t w) { return (w & E::TAKEN) != 0u; }
    __device__ void take(int t, uint32_t w) const { ew[t] = w | E::TAKEN; }
    __device__ int2 ord(int k) const { const int v = ol[k]; return make_int2(v & 0xff, v >> 8); }
    __device__ void set_ord(int k, int t, int l) const { ol[k] = (uint16_t)(t | (l << 8)); }
};

#if MACM_HUGE_BUILD
// An env's TCH x 32 bytes of touch_scratch: float2 n [TCH] ; float2 imp [TCH] ; u32 edge word a | b<<8 | taken<<31 [TCH] ;
// u16 next-of-a [TCH] ; u16 next-of-b [TCH] ; u16 slot [TCH] ; (2 x TCH bytes unused) ; u32 t | lvl<<16 [TCH].
// head / lastlvl are u16 per body in the env's NEW region (shared memory).
struct GmemStage {
    static constexpr int NONE = 0xffff;
    static constexpr uint32_t TAKEN = 0x80000000u;
    float2* n; float2* imp; uint32_t* ew; uint16_t* na; uint16_t* nb; uint16_t* slot; uint32_t* ol; uint16_t* head; uint16_t* lastlvl;
    template <int NC>
    __device__ GmemStage(const EnvS<NC>& S, const SimConst& P, int env)
    {
        unsigned char* p = P.scratch + (size_t)env * P.TCH * 32;
        const size_t T = (size_t)P.TCH;
        n = (float2*)p; imp = (float2*)(p + 8 * T); ew = (uint32_t*)(p + 16 * T); na = (uint16_t*)(p + 20 * T);
        nb = (uint16_t*)(p + 22 * T); slot = (uint16_t*)(p + 24 * T); ol = (uint32_t*)(p + 28 * T);
        head = reinterpret_cast<uint16_t*>(S.nw()); lastlvl = head + NC;
    }
    __device__ uint32_t edge(int t) const { return ew[t]; }
    __device__ static int a(uint32_t w) { return (int)(w & 0xffu); }
    __device__ static int b(uint32_t w) { return (int)((w >> 8) & 0xffu); }
    __device__ int next(uint32_t w, int t, int body) const { return a(w) == body ? na[t] : nb[t]; }
    __device__ void link(int t, uint32_t, int na_, int nb_) const { na[t] = (uint16_t)na_; nb[t] = (uint16_t)nb_; }
    __device__ static bool taken(uint32_t w) { return (w & TAKEN) != 0u; }
    __device__ void take(int t, uint32_t w) const { ew[t] = w | TAKEN; }
    __device__ int2 ord(int k) const { const uint32_t v = ol[k]; return make_int2((int)(v & 0xffffu), (int)(v >> 16)); }
    __device__ void set_ord(int k, int t, int l) const { ol[k] = (uint32_t)t | ((uint32_t)l << 16); }
};
#endif   // MACM_HUGE_BUILD

// Islands of the tc staged contacts: labels (seed body of each body's island), island order and levels.  Returns the
// number of levels.
template <int G, int APL, class St>
__device__ __forceinline__ int dense_islands(const Grp<G>& g, const EnvS<G * APL>& S, const St& st, int tc)
{
    uint32_t* label = S.label();
#pragma unroll
    for (int s = 0; s < APL; ++s) { st.lastlvl[g.gl + s * G] = 0; st.head[g.gl + s * G] = St::NONE; }
    g.sync();
    int L = 1;
    if (g.gl == 0) {
        uint8_t* stack = S.stack();
        AgentSet<G * APL> rem = {};   // bodies with a touching contact that are not in an island yet
        for (int t = 0; t < tc; ++t) {
            const uint32_t w = st.edge(t);
            const int a = St::a(w), b = St::b(w);
            st.link(t, w, st.head[a], st.head[b]);
            st.head[a] = t;
            st.head[b] = t;
            add_bit(rem, a);
            add_bit(rem, b);
        }
        int nord = 0;
        for (;;) {
            const int seed = highest_of(rem);   // the highest body left: Box2D walks its body list from the last-created body
            if (seed < 0) break;
            int sp = 0;
            stack[sp++] = (uint8_t)seed;
            drop_bit(rem, seed);
            while (sp > 0) {
                const int b = stack[--sp];
                label[b] = (uint32_t)seed;
                for (int t = st.head[b]; t != St::NONE;) {
                    const uint32_t w = st.edge(t);
                    const int ta = St::a(w), tb = St::b(w);
                    const int nx = st.next(w, t, b);
                    if (!St::taken(w)) {
                        st.take(t, w);
                        const int l = 1 + max((int)st.lastlvl[ta], (int)st.lastlvl[tb]);
                        st.set_ord(nord++, t, l);
                        st.lastlvl[ta] = l;
                        st.lastlvl[tb] = l;
                        L = max(L, l);
                        const int other = (ta == b) ? tb : ta;
                        if (bit_of(rem, other)) { drop_bit(rem, other); stack[sp++] = (uint8_t)other; }
                    }
                    t = nx;
                }
            }
        }
    }
    L = g.shfl(L, 0);
    g.sync();
    return L;
}

// b2ContactSolver ctor + InitializeVelocityConstraints (world normals at the pre-integration positions, impulses scaled
// by dtRatio), WarmStart and the velocity iterations level by level, then StoreImpulses to the HBM list.
template <int G, int APL, class St>
__device__ __forceinline__ void dense_solve_velocity(const Grp<G>& g, const EnvS<G * APL>& S, const St& st, const SimConst& P,
                                                     int tc, int nlev, float ratio, float2* c_imp)
{
    const float2* pos = S.pos(); float2* vel = S.vel();
    const float mass_n = P.normal_mass, mass_t = P.normal_mass;
    for (int t = g.gl; t < tc; t += G) {
        const uint32_t w = st.edge(t);
        const float2 pa = pos[St::a(w)], pb = pos[St::b(w)];
        float nx = 1.0f, ny = 0.0f;
        const float dx = pb.x - pa.x, dy = pb.y - pa.y;
        if ((dx * dx + dy * dy) > B2_EPSILON * B2_EPSILON) { nx = dx; ny = dy; b2normalize(nx, ny); }
        float2 im = make_float2(0.0f, 0.0f);
        if (P.warm_starting) { im = st.imp[t]; im.x = ratio * im.x; im.y = ratio * im.y; }
        st.n[t] = make_float2(nx, ny);
        st.imp[t] = im;
    }
    g.sync();
    for (int it = -1; it < P.vel_iters; ++it) {   // it == -1: WarmStart
        for (int lev = 1; lev <= nlev; ++lev) {
            for (int k = g.gl; k < tc; k += G) {
                const int2 o = st.ord(k);
                if (o.y != lev) continue;
                const int t = o.x;
                const uint32_t w = st.edge(t);
                const int a = St::a(w), b = St::b(w);
                const float2 n = st.n[t];
                float2 im = st.imp[t];
                float2 va = vel[a], vb = vel[b];
                if (it < 0) warm_start(n.x, n.y, im.x, im.y, P.inv_mass, va, vb);
                else solve_velocity(n.x, n.y, P.friction, mass_n, mass_t, P.inv_mass, im.x, im.y, va, vb);
                vel[a] = va; vel[b] = vb;
                st.imp[t] = im;
            }
            g.sync();
        }
    }
    for (int t = g.gl; t < tc; t += G) c_imp[st.slot[t]] = st.imp[t];
}

// The position iterations level by level; an island stops as soon as it is solved.  Leaves solved[] for the sleep pass.
template <int G, int APL, class St>
__device__ __forceinline__ void dense_solve_position(const Grp<G>& g, const EnvS<G * APL>& S, const St& st, const SimConst& P,
                                                     int tc, int nlev)
{
    float2* pos = S.pos();
    const uint32_t* label = S.label();
    uint8_t* isl_act = S.isl_act(); uint8_t* isl_bad = S.isl_bad();
#pragma unroll
    for (int s = 0; s < APL; ++s) { isl_act[g.gl + s * G] = 1; isl_bad[g.gl + s * G] = 0; }
    g.sync();
    for (int it = 0; it < P.pos_iters; ++it) {
        for (int lev = 1; lev <= nlev; ++lev) {
            for (int k = g.gl; k < tc; k += G) {
                const int2 o = st.ord(k);
                if (o.y != lev) continue;
                const uint32_t w = st.edge(o.x);
                const int a = St::a(w), b = St::b(w);
                const int isl = label[a];
                if (!isl_act[isl]) continue;
                float2 ca = pos[a], cb = pos[b];
                const float sep = solve_position(P.radius, P.k_sum, P.inv_mass, ca, cb);
                pos[a] = ca; pos[b] = cb;
                if (!(b2min(0.0f, sep) >= -3.0f * B2_LINEAR_SLOP)) isl_bad[isl] = 1;
            }
            g.sync();
        }
        bool any_bad = false;
#pragma unroll
        for (int s = 0; s < APL; ++s) {
            const int i = g.gl + s * G;
            const uint8_t bad = isl_bad[i];
            isl_act[i] = bad;
            isl_bad[i] = 0;
            any_bad |= bad != 0;
        }
        g.sync();
        if (!g.ballot(any_bad)) break;
    }
#pragma unroll
    for (int s = 0; s < APL; ++s) S.solved()[g.gl + s * G] = (P.pos_iters > 0) && !isl_act[g.gl + s * G];
    g.sync();
}

// The default kernels' entry points (shared-memory stage only): phase 5 calls the first two, phase 7 the third.
template <int G, int APL>
__device__ __noinline__ int dense_islands_smem(const Grp<G>& g, const EnvS<G * APL>& S, int tc)
{
    return dense_islands<G, APL>(g, S, SmemStage<G * APL>(S), tc);
}
template <int G, int APL>
__device__ __noinline__ void dense_solve_velocity_smem(const Grp<G>& g, const EnvS<G * APL>& S, const SimConst& P, int tc,
                                                       int nlev, float ratio, float2* c_imp)
{
    dense_solve_velocity<G, APL>(g, S, SmemStage<G * APL>(S), P, tc, nlev, ratio, c_imp);
}
template <int G, int APL>
__device__ __noinline__ void dense_solve_position_smem(const Grp<G>& g, const EnvS<G * APL>& S, const SimConst& P, int tc,
                                                       int nlev)
{
    dense_solve_position<G, APL>(g, S, SmemStage<G * APL>(S), P, tc, nlev);
}

#if MACM_HUGE_BUILD
// Phases 5 and 7 of the kernels built with the global-memory stage.  A full shared-memory stage (tc == TC) may be a
// truncated one: then every touching contact of the env's HBM list is staged in global memory, in birth order, and the
// env is solved from there.  Returns the number of levels, with bit 30 set when even the global stage was too small
// (the contacts beyond it are left out); MISC word 0 tells the position part which stage holds the env.  (The
// shared-memory stage is inlined here rather than called: fewer spills in this unit's step kernels, measured with ptxas.)
template <int G, int APL>
__device__ __noinline__ int dense_solve_velocity_huge(const Grp<G>& g, const EnvS<G * APL>& S, const SimConst& P, int env, int cnt,
                                                      int tc, float ratio, const uint32_t* c_ab, float2* c_imp)
{
    const GmemStage H(S, P, env);
    int ht = 0;
    bool overflow = false;
    if (tc == P.TC) {
        for (int base = 0; base < cnt; base += G) {
            const int k = base + g.gl;
            const uint32_t ab = k < cnt ? c_ab[k] : 0u;
            const bool touch = (ab >> 16) & 1u;
            const unsigned tm = g.ballot(touch);
            const int t = ht + __popc(tm & g.below());
            if (touch && t < P.TCH) {
                H.ew[t] = ab & 0xffffu;   // a | b<<8
                H.slot[t] = (uint16_t)k;
                // the first TC impulses were staged in shared memory by phase 2, the rest kept theirs in the HBM list
                H.imp[t] = t < P.TC ? S.t_imp()[t] : c_imp[k];
            }
            overflow |= touch && t >= P.TCH;
            ht += __popc(tm);
        }
    }
    const int gtc = ht <= P.TC ? 0 : min(ht, P.TCH);   // (uniform) 0: the shared-memory stage holds every touching contact
    if (g.gl == 0) S.misc()[0] = (uint32_t)gtc;
    if (!gtc) {
        const SmemStage<G * APL> st(S);
        const int nlev = dense_islands<G, APL>(g, S, st, tc);
        dense_solve_velocity<G, APL>(g, S, st, P, tc, nlev, ratio, c_imp);
        return nlev;
    }
    const int nlev = dense_islands<G, APL>(g, S, H, gtc);
    dense_solve_velocity<G, APL>(g, S, H, P, gtc, nlev, ratio, c_imp);
    return nlev | (g.ballot(overflow) ? (1 << 30) : 0);
}
template <int G, int APL>
__device__ __noinline__ void dense_solve_position_huge(const Grp<G>& g, const EnvS<G * APL>& S, const SimConst& P, int env, int tc,
                                                       int nlev)
{
    const int gtc = (int)S.misc()[0];
    if (gtc) dense_solve_position<G, APL>(g, S, GmemStage(S, P, env), P, gtc, nlev);
    else dense_solve_position<G, APL>(g, S, SmemStage<G * APL>(S), P, tc, nlev);
}
#endif   // MACM_HUGE_BUILD

// b2World::Step prologue of a world with new fixtures: FindNewContacts before Collide.  Runs on
// the first step after a reset only; out of line.
template <int G, int APL>
__device__ __noinline__ int fresh_world_contacts(const Grp<G>& g, const EnvS<G * APL>& S, const SimConst& P,
                                                 AgentSet<G * APL> alive, int cnt, uint32_t* c_ab, float2* c_imp,
                                                 bool& overflow)
{
    AgentSet<G * APL>* adj = S.adj();
    for (int base = 0; base < cnt; base += G) {
        const int k = base + g.gl;
        if (k < cnt) {
            const uint32_t ab = c_ab[k];
            or_bit(adj, ab & 0xff, (ab >> 8) & 0xff);
            or_bit(adj, (ab >> 8) & 0xff, ab & 0xff);
        }
    }
    g.sync();
    cnt = find_new_contacts<G, APL>(g, S, P, alive, alive, cnt, c_ab, c_imp, overflow);
#pragma unroll
    for (int s = 0; s < APL; ++s) adj[g.gl + s * G] = AgentSet<G * APL>{};
    g.sync();
    return cnt;
}

// The scripted actors of test_scripts/bots.py inside a rollout (the actions=None mode of mvmnt.py:86-92):
// the same rules and the same counter-based draws as macm_bot_kernel (macm_aux.cu).  tn = the agent's target
// node (r, theta) of the last observation.
__device__ __noinline__ uint32_t bot_action(const SimConst& P, const Rollout& R, float2 tn, int env, int i, int step)
{
    uint32_t a0 = 1, a1 = 1, a2 = 1, a3 = 0;
    switch (R.policy) {
        case MACM_BOT_FORWARD: a0 = 2; break;
        case MACM_BOT_ROTATE: a2 = 2; break;
        case MACM_BOT_DIAG: a0 = 2; a1 = 2; break;
        case MACM_BOT_RANDOM: {
            const uint64_t gi = (uint64_t)env * P.N + i;
            const Philox r(R.seed, gi + (uint64_t)P.env_base * P.N, 2u, (uint32_t)step);
            a0 = (uint32_t)(((uint64_t)r.c[0] * 3u) >> 32);
            a1 = (uint32_t)(((uint64_t)r.c[1] * 3u) >> 32);
            a2 = (uint32_t)(((uint64_t)r.c[2] * 3u) >> 32);
            a3 = P.kind == MACM_ENV_TDM ? (r.c[3] >> 31) : 0u;
            break;
        }
        case MACM_BOT_FLOCK: {
            const float th_sign = (tn.y > 0.0f) ? 1.0f : (tn.y < 0.0f ? -1.0f : 0.0f);
            const float ahead = fabsf(tn.y) < (float)(NP_PI / 4) ? 1.0f : 0.0f;
            if (!(tn.x < 1.0f)) { a2 = (uint32_t)(th_sign + 1.0f); a0 = (uint32_t)(ahead + 1.0f); }
            break;
        }
        case MACM_BOT_CIRCLE: {
            const uint64_t gi = (uint64_t)env * P.N + i;
            const Philox r(R.seed, gi + (uint64_t)P.env_base * P.N, 3u, (uint32_t)step);
            a0 = 2; a2 = (r.c[0] >> 31) ? 2u : 1u;
            break;
        }
        default: break;
    }
    return a0 | (a1 << 8) | (a2 << 16) | (a3 << 24);
}

// The combat actor (bots.py:3-16) inside a rollout: agent i's observation row (combat.py:206-227) is recomputed
// from the staged positions and angles with the arithmetic of tdm_observe, so the choice is the one
// macm_bot_kernel makes from the `obs` buffer: nearest enemy (lowest index among equal r), turn towards it,
// walk when it is within +-36 degrees, strike inside 3 m.
template <int W>
__device__ __noinline__ uint32_t combat_action(const float2* pos, const float* angs, const uint8_t* team, int N,
                                               Bits<W> alive, int i)
{
    uint32_t a0 = 1, a2 = 1, a3 = 0;
    if (i < N && bit_of(alive, i)) {
        const float2 p = pos[i];
        const int ti = team[i];
        float br = 0.0f, bdx = 0.0f, bdy = 0.0f;
        bool found = false;
        for (int j = 0; j < N; ++j) {
            if (j == i || !bit_of(alive, j) || team[j] == ti) continue;
            const float2 q = pos[j];
            const float dx = q.x - p.x, dy = q.y - p.y;
            const float r = out_sqrtf(dx * dx + dy * dy);
            if (!found || r < br) { br = r; bdx = dx; bdy = dy; found = true; }
        }
        if (found) {
            const float th = wrap_pi_f(fast_atan2f(bdy, bdx) - angs[i]);
            a0 = (fabs((double)th) < NP_PI / 5) ? 2u : 1u;
            a2 = th > 0.0f ? 2u : (th < 0.0f ? 0u : 1u);
            a3 = br < 3.0f ? 1u : 0u;
        }
    }
    return a0 | (1u << 8) | (a2 << 16) | (a3 << 24);
}

// ------------------------------------------------------------------------------------------
// the step kernel
// ------------------------------------------------------------------------------------------
// MODE 0: one step per launch (macm_step); every rollout argument folds away at compile time.
// MODE 1: R.K steps per launch (macm_rollout), the env's bodies staying in registers / shared memory.
// MODE 2: one step per launch whose outputs ALSO go to the caller's per-step arrays (macm_rollout with n_steps = 1
//         and given actions -- the shape gym_macm.dist.PeerGather uses to store into the learner's memory): the
//         single-step code plus the second stores, none of the loop-carried state of MODE 1.
// widest block of a shape: 28 warps of one env each; envs of 65..128 agents (four agents per lane) take 14 warps with
// twice the registers per thread
__host__ __device__ constexpr int shape_max_threads(int G, int APL) { return APL == 4 ? MACM_WIDE_THREADS / 2 : MACM_WIDE_THREADS; }

template <int G, int APL, int KIND, int MODE>
__global__ void __launch_bounds__(shape_max_threads(G, APL), 1) macm_step_kernel(const __grid_constant__ SimConst P,
                                                        const void* __restrict__ actions,
                                                        const __grid_constant__ Rollout R_)
{
    // the single-step kernel sees compile-time constants instead of the rollout arguments
    constexpr bool ROLL = MODE == 1;   // the multi-step loop with its parked state
    struct RollView {
        const Rollout& r;
        __device__ int K() const { return MODE == 1 ? r.K : 1; }
        __device__ int policy() const { return MODE == 1 ? r.policy : -1; }
        __device__ int sync() const { return MODE == 1 ? r.sync : 0; }
        __device__ float* obs() const { return MODE ? r.obs : nullptr; }
        __device__ int* nn_idx() const { return MODE ? r.nn_idx : nullptr; }
        __device__ float* rewards() const { return MODE ? r.rewards : nullptr; }
        __device__ uint8_t* collided() const { return MODE ? r.collided : nullptr; }
        __device__ uint8_t* done() const { return MODE ? r.done : nullptr; }
    };
    const RollView R{R_};
    constexpr int NC = G * APL;
    constexpr int GPW = 32 / G;
    constexpr bool TDM = KIND == MACM_ENV_TDM;
    constexpr bool HUGE = MACM_HUGE_BUILD;   // this translation unit's kernels carry the global-memory touching stage
    using EWT = EW<NC>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Grp<G> g;
    const int slot_in_block = (threadIdx.x >> 5) * GPW + (threadIdx.x & 31) / G;
    const int slot = blockIdx.x * (blockDim.x / 32) * GPW + slot_in_block;
    // One block per SM: the sin/cos table of the action decode (library-owned, written once at
    // macm_create) is copied to shared memory before anything else -- under programmatic dependent launch
    // that happens while the previous kernel drains, and phase 1 no longer waits for L2.
    const double2* sincos_tab = P.sincos_tab;
    if (blockDim.x > 128) {
        double2* tab_s = reinterpret_cast<double2*>(smem_raw + (size_t)(blockDim.x / 32) * GPW * Lay<NC>::bytes(P.TC));
        for (int k = threadIdx.x; k < MACM_TABLE_BYTES / 16; k += blockDim.x) tab_s[k] = __ldg(&P.sincos_tab[k]);
        __syncthreads();
        sincos_tab = tab_s;
    }
    if (slot >= P.E) return;  // whole group leaves together
    unsigned long long tr_t0 = 0, tr_c0 = 0;
    const int N = P.N;
    EnvS<NC> S;
    S.TC = P.TC;
    S.base = smem_raw + (size_t)slot_in_block * Lay<NC>::bytes(P.TC);

    float2* pos = S.pos(); float2* vel = S.vel(); float4* fat = S.fat();
    typedef AgentSet<NC> ASet;
    ASet* adj = S.adj();
    uint32_t* label = S.label();
    uint32_t* tmask = S.tmask();

    // Programmatic dependent launch: this grid may have been scheduled while the previous kernel of
    // the stream was still draining (its blocks take the SM slots as they free up).  No value is read
    // from global memory before the wait; the env's lines are only pulled towards L2 (the coherence
    // point, so a line the predecessor is still writing cannot go stale there), which takes the HBM
    // latency of the state off the critical path whenever there is a predecessor to overlap with.
    // (small-env shapes only: their launches are several waves of 128-thread blocks, and a block of a later wave gains
    //  nothing from pulling lines it loads a few instructions later -- config 3: 27.5 -> 25.5 us.  The one-env-per-warp
    //  kernel keeps the unconditional form: the same test there cost its zero-spill register allocation, +0.4 us.)
    if (G == 32 || (int)blockIdx.x < P.first_wave) {
        // one line per lane: 8 lanes on posvel, 8 on the fat AABBs (or the TDM state after the first 4), 4 on
        // angle/sleep, 2 on the actions, 1 + 2 on the head of the contact list, then the per-env scalars.
        // (Everything before griddepcontrol.wait runs while the predecessor drains: a branch-free / table-driven
        // version of this ladder, 25 instead of 120 instructions, measured SLOWER -- 20.8 against 18.8 us per step --
        // because its indexed constant loads delayed the prefetches; profiles/README.md, r2 finding 2.)
        const int env_ = slot, l = g.gl;
        const size_t a0 = (size_t)env_ * P.N;
        const int abytes = (TDM || P.action_mode == MACM_ACTION_DISCRETE) ? 4 : 8;
        const char* p = nullptr;
        int off = 0, lim = 0;
        if (l < 8) { p = (const char*)(P.posvel + a0); off = l * 128; lim = P.N * 16; }
        else if (l < 16) { p = (const char*)(P.fat + a0); off = (l - 8) * 128; lim = P.N * 16; }
        else if (l < 20) { p = (const char*)(P.angsleep + a0); off = (l - 16) * 128; lim = P.N * 8; }
        else if (l < 24) { if (actions) { p = (const char*)actions + a0 * abytes; off = (l - 20) * 128; lim = P.N * abytes; } }
        else if (l < 25) { p = (const char*)(P.c_ab + (size_t)env_ * P.C); lim = 1; }
        else if (l < 27) { p = (const char*)(P.c_imp + (size_t)env_ * P.C); off = (l - 25) * 128; lim = 256; }
        else if (l < 28) { p = (const char*)(P.env_state + env_); lim = 1; }
        else if (l < 29) { p = (const char*)(P.c_cnt + env_); lim = 1; }
        else if (l < 30) { if (!TDM) { p = (const char*)(P.targets + (size_t)env_ * P.T); lim = 1; } }
        if (G == 32 && off < lim) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + off));
        if (G == 32 && TDM) prefetch_l2<G>(g.gl, P.tdm + a0, P.N * 16);
        if (G < 32) {   // several envs per warp: a few lines each
            prefetch_l2<G>(g.gl, P.posvel + a0, P.N * 16);
            prefetch_l2<G>(g.gl, P.fat + a0, P.N * 16);
            prefetch_l2<G>(g.gl, P.angsleep + a0, P.N * 8);
        }
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (P.trace) { asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_t0)); tr_c0 = clock64(); }
    const int env = slot;
    uint32_t* c_ab = P.c_ab + (size_t)env * P.C;
    float2* c_imp = P.c_imp + (size_t)env * P.C;

    // ---- phase 0: load state ---------------------------------------------------------------
    float2 c[APL], v[APL], F[APL];
    float ang[APL], slp[APL];
    float4 fatr[APL];
    bool valid[APL];
    uint32_t act_raw[APL];
    const int4 es0 = P.env_state[env];
    int step_cnt = es0.x, eflags = es0.y, winner = es0.w;   // b2World step count, MACM_ENV_* bits, TDM winner
    int cnt = P.c_cnt[env];
    // first chunk of the contact list, fetched together with the state (one HBM round trip less)
    uint32_t pre_ab = 0u;
    float2 pre_imp = make_float2(0.0f, 0.0f);
    if (g.gl < P.C) { pre_ab = c_ab[g.gl]; pre_imp = c_imp[g.gl]; }
    // TDM per-agent host state (combat.Agent): health, cool-downs (steps left), alive, hits taken
    float health[APL];
    int cd_atk[APL], cd_mov[APL], hits[APL];
    bool was_alive[APL];
    int team[APL];
    float2 tg0[APL];   // the agent's target, on its way to shared memory
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        valid[s] = i < N;
        team[s] = (TDM && valid[s]) ? P.team[i] : 0;
        const size_t gi = (size_t)env * N + (valid[s] ? i : 0);
        const float4 pv = P.posvel[gi];
        const float2 as = P.angsleep[gi];
        fatr[s] = P.fat[gi];
        c[s] = make_float2(pv.x, pv.y); v[s] = make_float2(pv.z, pv.w); ang[s] = as.x; slp[s] = as.y;
        was_alive[s] = valid[s];
        if (TDM) {
            const float4 td = P.tdm[gi];
            health[s] = td.x; cd_atk[s] = __float_as_int(td.y); cd_mov[s] = __float_as_int(td.z);
            const int w = __float_as_int(td.w);
            was_alive[s] = valid[s] && (w & 1);
            hits[s] = w >> 8;
        }
        if (!valid[s]) {  // padding agents: parked far away
            c[s] = make_float2(3.0e30f, 3.0e30f); v[s] = make_float2(0.0f, 0.0f);
            fatr[s] = make_float4(3.0e30f, 3.0e30f, 3.0e30f, 3.0e30f);
        }
        // (one target: no index to fetch first -- one dependent global load less at the head of the step)
        if (!TDM) tg0[s] = P.targets[(size_t)env * P.T + (P.T == 1 ? 0 : (int)P.target_idx[valid[s] ? i : 0])];
        if (!TDM && ROLL) S.tgt()[i] = tg0[s];   // (a rollout stages it before its loop)
        // the flock actor steers by the target node of the last observation (bots.py:37-61)
        if (!TDM && R.policy() == MACM_BOT_FLOCK && valid[s]) {
            const float4 o4 = reinterpret_cast<const float4*>(P.obs)[gi];   // fp32 polar only (macm_rollout checks)
            reinterpret_cast<float2*>(S.nw())[i] = make_float2(o4.z, o4.w);
        }
    }
    const bool discrete = TDM || P.action_mode == MACM_ACTION_DISCRETE;
    const size_t EN = (size_t)P.E * N;
    int tc = 0, nlev = 0;
    bool multi = false;

    // ---- K steps of this env; its state stays in registers / shared memory between them -------------
#pragma unroll 1
    for (int ks = 0; ks < R.K(); ++ks) {
    const bool last = ks == R.K() - 1;
    ASet alive = {};   // bodies that are active (have a proxy) during this step
    // The block's warps start every R.sync()-th step together.  Measured (profiles/README.md, finding 8): the hot
    // path is ~48 KB of straight-line code; warps that drift apart each stream it from the GPC-level instruction
    // cache on their own, which saturates (gcc requests 83 % of peak, "no instruction" the top stall) -- in step
    // they share every fetched line.
    if (R.sync() > 0 && ks > 0 && (ks % R.sync()) == 0) __syncthreads();
    g.sync();   // the previous step's observation pass has finished reading the staging arrays
    ASet alive0 = {};   // (combat actor) who is in the observation the actors decide on
    if (ROLL && TDM && R.policy() == MACM_BOT_COMBAT) {
        if (ks == 0) {   // later steps: positions and angles are staged since the previous step's phases 7 and 11
#pragma unroll
            for (int s = 0; s < APL; ++s) { pos[g.gl + s * G] = c[s]; S.ang()[g.gl + s * G] = ang[s]; }
        }
#pragma unroll
        for (int s = 0; s < APL; ++s) {
            const unsigned bm = g.ballot(was_alive[s]);
            put_slot<G>(alive0, s, bm);
        }
        g.sync();
    }
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        const size_t gi = (size_t)env * N + (valid[s] ? i : 0);
        if (ROLL && ks > 0) {   // parked before the previous step's observation pass (see there)
            v[s] = vel[i];
            fatr[s] = reinterpret_cast<const float4*>(S.t_n())[i];
            slp[s] = reinterpret_cast<const float*>(reinterpret_cast<const float4*>(S.t_n()) + NC)[i];
        }
        // discrete action word, fetched with the state (first step) / one step ahead into L2 (later steps)
        act_raw[s] = 0u;
        if (discrete && valid[s]) {
            if (!ROLL || actions) {
                const uint32_t* aw = reinterpret_cast<const uint32_t*>(actions) + (size_t)ks * EN + gi;
                act_raw[s] = *aw;
                if (!last) asm volatile("prefetch.global.L2 [%0];" ::"l"(aw + EN));
            } else if (TDM && R.policy() == MACM_BOT_COMBAT) {
                act_raw[s] = combat_action(pos, S.ang(), P.team, N, alive0, i);
            } else {
                act_raw[s] = bot_action(P, R_, reinterpret_cast<const float2*>(S.nw())[i], env, i, step_cnt);
            }
        }
    }

    PHASE_STAMP(0);
    // ---- phase 1: actions -> angle, force (mvmnt.py:97-129 / combat.py:121-155), float64 like the reference
    bool attack[APL];
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        F[s] = make_float2(0.0f, 0.0f);
        attack[s] = false;
        if (!was_alive[s]) continue;
        const size_t gi = (size_t)env * N + i;
        if (TDM || P.action_mode == MACM_ACTION_DISCRETE) {
            const uint32_t act = act_raw[s];
            const int a0 = (int)(act & 0xff) - 1, a1 = (int)((act >> 8) & 0xff) - 1, a2 = (int)((act >> 16) & 0xff) - 1;
            // body.angle = body.angle + (a2-1) * rotation_speed * (1/hz)   -> SetTransform rounds to fp32
            float af = (float)((double)ang[s] + (double)a2 * P.rot_step);
            if (fabs((double)af) > NP_PI) {
                const double a = (double)af;
                const double sg = (a > 0.0) ? 1.0 : -1.0;
                af = (float)(a - sg * (2 * NP_PI));
            }
            ang[s] = af;
            // np.cos(angle), np.sin(angle), np.cos(angle + np.pi/2), np.sin(angle + np.pi/2) in float64.
            // t = fl(A + pi/2) = (A + pi/2) + d exactly, with d from the rounding error of the sum and
            // the tail of pi/2, so cos t = -sin(A + d) = -(sin A + d cos A), sin t = cos A - d sin A.
            double s1, c1;
            sincos_f32arg(sincos_tab, af, s1, c1);
            const double A = (double)af, H = NP_PI / 2;
            const double t = A + H, bb = t - A;
            const double err = (A - (t - bb)) + (H - bb);          // A + H == t + err exactly (TwoSum)
            const double d = -(err + 6.123233995736766e-17);       // pi/2 = H + 6.1232...e-17
            const double c2 = -fma(d, c1, s1), s2 = fma(-d, s1, c1);
            const double cc = (a0 != 0 && a1 != 0) ? P.diag : 1.0;
            double force = P.force;
            if (TDM) force = cd_mov[s] > 0 ? P.force_pen : P.force;   // Agent.force (combat.py:46-49)
            F[s].x = (float)((c1 * (double)a0 + c2 * (double)a1) * cc * force);
            F[s].y = (float)((s1 * (double)a0 + s2 * (double)a1) * cc * force);
            if (TDM) {
                // attack (combat.py:142-155): ray from the centre, melee_range along the heading
                bool started = false;
                if (cd_atk[s] <= 0) {
                    if ((act >> 24) & 0xff) {
                        attack[s] = true;
                        started = true;
                        cd_atk[s] = P.cd_atk_steps;
                        cd_mov[s] = P.cd_mov_steps;
                        const float dx = (float)(P.melee_range * c1), dy = (float)(P.melee_range * s1);
                        reinterpret_cast<float2*>(S.nw())[i] = make_float2(c[s].x + dx, c[s].y + dy);
                    }
                } else {
                    cd_atk[s] -= 1;
                }
                if ((P.flags & MACM_FLAG_REPAIR_MOV_COOLDOWN) && !started && cd_mov[s] > 0) cd_mov[s] -= 1;
            }
        } else {
            const float2 ac = reinterpret_cast<const float2*>(actions)[(size_t)ks * EN + gi];
            double x = (double)ac.x, y = (double)ac.y;
            if ((x * x + y * y) > 1) {  // bug-compatible with mvmnt.py:124-126
                x = sqrt(x * x / (x * x + y * y));
                y = sqrt(y * y / (x * x + y * y));
            }
            F[s].x = (float)(x * P.force);
            F[s].y = (float)(y * P.force);
        }
    }
    // The bodies reach shared memory only now: phase 1 needs nothing but the angle and the action word, so the
    // rest of the state (positions, fat AABBs, contact list head, target) is still arriving from L2 while the
    // float64 action decode runs -- the whole batch loads its state at the same moment and the L2 is the queue.
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        pos[i] = c[s];
        fat[i] = fatr[s];
        adj[i] = ASet{};
        S.tmask()[i] = 0u;
        if (!TDM && !ROLL) S.tgt()[i] = tg0[s];
    }
    g.sync();

    PHASE_STAMP(1);
    // ---- phase 1b (TDM): closest-hit ray casts, health, deaths (combat.py:141-165, cm_framework.py:56-86)
    bool now_alive[APL];
#pragma unroll
    for (int s = 0; s < APL; ++s) now_alive[s] = was_alive[s];
    if (TDM) {
        unsigned am[APL];
        bool any_attack = false;
#pragma unroll
        for (int s = 0; s < APL; ++s) { am[s] = g.ballot(attack[s]); any_attack |= am[s] != 0u; }
        if (any_attack) {
            const float2* ray = reinterpret_cast<const float2*>(S.nw());
#pragma unroll
            for (int w = 0; w < APL; ++w) {
                for (unsigned mm = am[w]; mm; mm &= mm - 1) {
                    const int m = w * G + __ffs((int)mm) - 1;
                    const float2 p1 = pos[m], p2 = ray[m];
                    const float4 r4 = make_float4(p1.x, p1.y, p2.x, p2.y);
                    // b2CircleShape::RayCast against every proxy; keep the smallest fraction,
                    // lowest index among equal fractions
                    unsigned fk[APL];
                    unsigned key = 0xffffffffu;
#pragma unroll
                    for (int s = 0; s < APL; ++s) {
                        fk[s] = 0xffffffffu;
                        if (!was_alive[s]) continue;
                        const float sx = r4.x - c[s].x, sy = r4.y - c[s].y;
                        const float bq = (sx * sx + sy * sy) - P.radius * P.radius;
                        const float rx = r4.z - r4.x, ry = r4.w - r4.y;
                        const float cq = sx * rx + sy * ry;
                        const float rr = rx * rx + ry * ry;
                        const float sigma = cq * cq - rr * bq;
                        if (sigma < 0.0f || rr < B2_EPSILON) continue;
                        float a = -(cq + sqrtf(sigma));
                        if (0.0f <= a && a <= 1.0f * rr) {
                            a /= rr;
                            fk[s] = __float_as_uint(a);   // a >= 0: bit order == value order
                            key = min(key, fk[s]);
                        }
                    }
                    const unsigned kmin = g.reduce_min(key);
                    if (kmin != 0xffffffffu) {
                        // lowest agent index with that fraction
                        unsigned mine = 0xffffffffu;
#pragma unroll
                        for (int s = APL - 1; s >= 0; --s)
                            if (fk[s] == kmin) mine = g.gl + s * G;
                        const unsigned victim = g.reduce_min(mine);
#pragma unroll
                        for (int s = 0; s < APL; ++s) if ((unsigned)(g.gl + s * G) == victim) hits[s] += 1;
                    }
                }
            }
        }
        // health -= melee_dmg per hit, in the reference's float64 (combat.py:153); deaths (combat.py:157-165)
#pragma unroll
        for (int s = 0; s < APL; ++s) {
            if (!was_alive[s]) continue;
            double h = (double)P.init_health;
            for (int k = 0; k < hits[s]; ++k) h -= P.melee_dmg_d;
            health[s] = (float)h;
            if (h <= 0) now_alive[s] = false;   // body.active = False: proxy and contacts go at once
        }
        g.sync();
    }
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const unsigned bm = g.ballot(now_alive[s]);
        put_slot<G>(alive, s, bm);
    }

    bool overflow_c = false, overflow_t = false;

    PHASE_STAMP(2);
    // ---- phase 2a: new fixtures -> FindNewContacts before Collide (b2World::Step prologue) ----
    if (eflags & MACM_ENV_FRESH) cnt = fresh_world_contacts<G, APL>(g, S, P, alive, cnt, c_ab, c_imp, overflow_c);

    // ---- phase 2: b2ContactManager::Collide --------------------------------------------------
    // destroy contacts whose fat AABBs stopped overlapping (or whose body was deactivated),
    // narrowphase the rest, compact in place (birth order is preserved), stage the touching ones
    tc = 0;
    multi = false;   // some body has two touching contacts: islands are more than pairs
    {
        float2* t_imp = S.t_imp();
        uint32_t* t_ew = S.t_ew();
        uint16_t* t_slot = S.t_slot();
        int w = 0;
        bool dup = false;
        for (int base = 0; base < cnt; base += G) {
            const int k = base + g.gl;
            const bool in = k < cnt;
            uint32_t ab = 0;
            float2 imp = make_float2(0.0f, 0.0f);
            if (in) {
                if (base == 0 && ks == 0 && !(eflags & MACM_ENV_FRESH)) { ab = pre_ab; imp = pre_imp; }
                else { ab = c_ab[k]; imp = c_imp[k]; }
            }
            g.sync();  // every lane holds its record before any lane compacts over it
            const int a = ab & 0xff, b = (ab >> 8) & 0xff;
            bool keep = in && aabb_overlap(fat[a], fat[b]);
            if (TDM) keep = keep && bit_of(alive, a) && bit_of(alive, b);
            bool touch = false;
            if (keep) {
                const float2 pa = pos[a], pb = pos[b];
                const float dx = pb.x - pa.x, dy = pb.y - pa.y;
                touch = !((dx * dx + dy * dy) > P.rsum2);
            }
            const unsigned km = g.ballot(keep), tm = g.ballot(touch);
            if (keep) {
                const int p = w + __popc(km & g.below());
                const bool was = (ab >> 16) & 1;
                const float nI = (touch && was) ? imp.x : 0.0f, tI = (touch && was) ? imp.y : 0.0f;
                c_ab[p] = (uint32_t)a | ((uint32_t)b << 8) | ((uint32_t)touch << 16);
                const int tp = tc + __popc(tm & g.below());
                // touching contacts get their impulses from StoreImpulses after the solver
                if (!touch || tp >= P.TC) c_imp[p] = make_float2(nI, tI);
                or_bit(adj, a, b);
                or_bit(adj, b, a);
                if (touch && tp < P.TC) {
                    t_ew[tp] = (uint32_t)a | ((uint32_t)b << EWT::SH_B);
                    t_imp[tp] = make_float2(nI, tI);
                    t_slot[tp] = (uint16_t)p;
                    // the body's set of touching contacts; does any body carry two?
                    if (tp < 32) {
                        const uint32_t oa = atomicOr(&tmask[a], 1u << tp);
                        const uint32_t ob = atomicOr(&tmask[b], 1u << tp);
                        dup |= (oa | ob) != 0u;
                    }
                }
            }
            w += __popc(km);
            tc += __popc(tm);
        }
        cnt = w;
        if (tc > P.TC) { overflow_t = !HUGE; tc = P.TC; }   // (HUGE: the global-memory stage takes the env)
        multi = g.ballot(dup) != 0u;
    }

    PHASE_STAMP(3);
    // ---- phase 3: integrate velocities (b2Island::Solve, first loop) -------------------------
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        if (now_alive[s]) {
            // v += h * (gravityScale * gravity + invMass * force); v *= damping
            v[s].x += P.h * (P.inv_mass * F[s].x);
            v[s].y += P.h * (P.inv_mass * F[s].y);
            v[s].x *= P.damp;
            v[s].y *= P.damp;
        }
        vel[i] = v[s];
        label[i] = (uint32_t)i;
        // an island without contacts passes its first position iteration (minSeparation = 0)
        S.solved()[i] = P.pos_iters > 0;
    }
    g.sync();

    PHASE_STAMP(4);
    // ---- phase 4: islands (b2World::Solve) ---------------------------------------------------------
    // Box2D seeds islands from the body list (last-created body first), pops a stack, walks each
    // body's contact edges newest-first and solves an island's contacts in the order it added them.
    // Islands share no body, so each one is replayed and solved by ONE lane, sequentially, in exactly
    // that order -- no ordering between islands is needed and no barrier inside the solver.
    //   * no body with two touching contacts (the usual case): islands are the pairs themselves,
    //     contact k lives in the registers of lane k for the whole solve;
    //   * otherwise (tc <= G): label propagation finds each island's seed (its highest body index),
    //     the k-th seed goes to lane k, which runs the DFS over the bodies' touching-contact sets
    //     (bit t = staged contact t, highest = newest) and threads the contacts into a list;
    //   * dense piles (tc > G): one lane replays the DFS for the whole world and the contacts are
    //     level-scheduled across lanes (dense_* above, out of line).
    const bool big = tc > G;
    const bool has = !big && g.gl < tc;
    nlev = 0;
    int ka = 0, kb = 0;
    float knx = 1.0f, kny = 0.0f, knI = 0.0f, ktI = 0.0f;
    int ohead = EW_NONE, oseed = 0;     // multi: first contact of this lane's island, its seed body
    // inv_dt0 == 0 on a world's first step -> dtRatio 0
    const float ratio = (step_cnt == 0) ? 0.0f : P.dt_ratio;
#if MACM_HUGE_BUILD
    // a dense pile's level count, phase 5 to 7 (nlev stays 0 in this unit: live for the whole step it costs spills)
    int hlev = 0;
#endif

    // ---- phase 5: contact solver, velocity part -------------------------------------------------
    if (big) {
#if MACM_HUGE_BUILD
        hlev = dense_solve_velocity_huge<G, APL>(g, S, P, env, cnt, tc, ratio, c_ab, c_imp);
        if (hlev >> 30) { overflow_t = true; hlev &= 0xffff; }
#else
        nlev = dense_islands_smem<G, APL>(g, S, tc);
        dense_solve_velocity_smem<G, APL>(g, S, P, tc, nlev, ratio, c_imp);
#endif
    } else if (tc > 0) {
        const float mass_n = P.normal_mass, mass_t = P.normal_mass;
        uint32_t* t_ew = S.t_ew();
        // b2ContactSolver ctor + InitializeVelocityConstraints: world manifold at the
        // pre-integration positions, impulses scaled by dtRatio
        if (has) {
            const uint32_t ew = t_ew[g.gl];
            ka = EWT::a(ew); kb = EWT::b(ew);
            const float2 pa = pos[ka], pb = pos[kb];
            const float dx = pb.x - pa.x, dy = pb.y - pa.y;
            // b2DistanceSquared(pointA, pointB) is (A - B).(A - B); squares are sign-blind
            if ((dx * dx + dy * dy) > B2_EPSILON * B2_EPSILON) { knx = dx; kny = dy; b2normalize(knx, kny); }
            if (P.warm_starting) { const float2 im = S.t_imp()[g.gl]; knI = ratio * im.x; ktI = ratio * im.y; }
        }
        if (!multi) {
            // independent contacts: warm start + all iterations without leaving registers
            if (has) {
                float2 va = vel[ka], vb = vel[kb];
                warm_start(knx, kny, knI, ktI, P.inv_mass, va, vb);
                for (int it = 0; it < P.vel_iters; ++it)
                    solve_velocity(knx, kny, P.friction, mass_n, mass_t, P.inv_mass, knI, ktI, va, vb);
                vel[ka] = va; vel[kb] = vb;
                label[ka] = (uint32_t)kb;   // the pair's island is seeded by its higher index
                oseed = kb;
                // StoreImpulses -> manifold (next step's warm start)
                c_imp[S.t_slot()[g.gl]] = make_float2(knI, ktI);
            }
            g.sync();
        } else {
            float2* t_n = S.t_n(); float2* t_imp = S.t_imp();
            // Islands = connected sets of touching contacts.  Contact t lives in lane t; the contacts
            // next to it are the touching-contact sets of its two bodies.  The sets are closed under
            // "shares a body" with shuffles (islands are a few contacts: one or two rounds), together
            // with the highest body index of the island, which is Box2D's seed for it.
            uint32_t cset = 0u;
            int seed = 0;
            if (has) {
                t_n[g.gl] = make_float2(knx, kny);
                t_imp[g.gl] = make_float2(knI, ktI);
                cset = tmask[ka] | tmask[kb];
                seed = kb;   // a < b
            }
            for (;;) {
                uint32_t acc = cset;
                int top = seed;
                uint32_t todo = cset & ~(1u << g.gl);
                while (g.ballot(todo != 0u)) {
                    const int u = todo ? (__ffs((int)todo) - 1) : g.gl;
                    const uint32_t cu = (uint32_t)g.shfl((int)cset, u);
                    const int su = g.shfl(seed, u);
                    acc |= cu;
                    top = max(top, su);
                    todo &= todo - 1u;
                }
                const bool changed = acc != cset || top != seed;
                cset = acc; seed = top;
                if (!g.ballot(changed)) break;
            }
            nlev = 0;
            if (has) { label[ka] = (uint32_t)seed; label[kb] = (uint32_t)seed; }
            g.sync();
#ifdef MACM_PHASE_TRACE
            if (P.trace && g.gl == 0) P.trace[(size_t)env * 16 + 13] = clock64() - tr_c0;
            unsigned long long dfs_done = 0;
#endif
            // the lane of an island's first contact replays Box2D's DFS for it and then solves it
            if (has && (__ffs((int)cset) - 1) == g.gl) {
                oseed = seed;
                uint8_t* nxt = S.stack();
                uint32_t taken = 0u;
                ASet vis = {};   // bodies pushed so far
                int top = oseed, otail = EW_NONE;
                uint32_t otail_ew = 0u;
                nxt[oseed] = EW_NONE;
                add_bit(vis, oseed);
                while (top != EW_NONE) {
                    const int b = top;
                    top = nxt[b];
                    for (uint32_t m = tmask[b] & ~taken; m;) {
                        const int t = 31 - __clz((int)m);   // newest edge first
                        m &= ~(1u << t);
                        taken |= 1u << t;
                        const uint32_t ew = t_ew[t] & EWT::AB;
                        if (otail == EW_NONE) ohead = t; else t_ew[otail] = otail_ew | ((uint32_t)t << EWT::SH_NA);
                        otail = t; otail_ew = ew;
                        const int other = (EWT::a(ew) == b) ? EWT::b(ew) : EWT::a(ew);
                        if (!bit_of(vis, other)) {
                            add_bit(vis, other);
                            nxt[other] = (uint8_t)top;
                            top = other;
                        }
                    }
                }
                t_ew[otail] = otail_ew | ((uint32_t)EW_NONE << EWT::SH_NA);
#ifdef MACM_PHASE_TRACE
                dfs_done = clock64() - tr_c0;
#endif
                // b2ContactSolver::WarmStart, then the velocity iterations, in island order.  The next
                // contact's record is fetched while the current one is being solved.
                const uint32_t ew_head = t_ew[ohead];
                const float2 n_head = t_n[ohead];
                for (int it = -1; it < P.vel_iters; ++it) {
                    int t = ohead;
                    uint32_t ew = ew_head;
                    float2 n = n_head, im = t_imp[t];
                    for (;;) {
                        const int a = EWT::a(ew), b = EWT::b(ew), tn = EWT::na(ew);
                        float2 va = vel[a], vb = vel[b];
                        uint32_t ew2 = 0u;
                        float2 n2 = make_float2(0.0f, 0.0f), im2 = n2;
                        if (tn != EW_NONE) { ew2 = t_ew[tn]; n2 = t_n[tn]; im2 = t_imp[tn]; }
                        if (it < 0) warm_start(n.x, n.y, im.x, im.y, P.inv_mass, va, vb);
                        else solve_velocity(n.x, n.y, P.friction, mass_n, mass_t, P.inv_mass, im.x, im.y, va, vb);
                        vel[a] = va; vel[b] = vb;
                        t_imp[t] = im;
                        if (tn == EW_NONE) break;
                        t = tn; ew = ew2; n = n2; im = im2;
                    }
                }
            }
            g.sync();
#ifdef MACM_PHASE_TRACE
            {
                const unsigned lo = __reduce_max_sync(g.mask, (unsigned)dfs_done);
                if (P.trace && g.gl == 0) P.trace[(size_t)env * 16 + 14] = lo;
            }
#endif
            // StoreImpulses -> manifold (next step's warm start)
            if (has) c_imp[S.t_slot()[g.gl]] = t_imp[g.gl];
        }
    }
    PHASE_STAMP(5);
    // ---- phase 6: integrate positions ------------------------------------------------------------
    float2 c0[APL];
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        c0[s] = c[s];
        if (!now_alive[s]) continue;
        float2 w = vel[i];
        const float trx = P.h * w.x, try_ = P.h * w.y;
        if ((trx * trx + try_ * try_) > B2_MAX_TRANSLATION * B2_MAX_TRANSLATION) {
            const float ratio = B2_MAX_TRANSLATION / sqrtf(trx * trx + try_ * try_);
            w.x *= ratio; w.y *= ratio;
        }
        c[s].x += P.h * w.x;
        c[s].y += P.h * w.y;
        v[s] = w;
    }
    g.sync();
#pragma unroll
    for (int s = 0; s < APL; ++s) pos[g.gl + s * G] = c[s];
    g.sync();

    PHASE_STAMP(6);
    // ---- phase 7: contact solver, position part (each island stops as soon as it is solved) -------
    if (big) {
#if MACM_HUGE_BUILD
        dense_solve_position_huge<G, APL>(g, S, P, env, tc, hlev);
#else
        dense_solve_position_smem<G, APL>(g, S, P, tc, nlev);
#endif
#pragma unroll
        for (int s = 0; s < APL; ++s) c[s] = pos[g.gl + s * G];
    } else if (tc > 0) {
        if (!multi) {
            if (has) {
                float2 ca = pos[ka], cb = pos[kb];
                bool ok = false;
                for (int it = 0; it < P.pos_iters && !ok; ++it) {
                    const float sep = solve_position(P.radius, P.k_sum, P.inv_mass, ca, cb);
                    // solved once min(0, separations) >= -3 * linearSlop
                    ok = b2min(0.0f, sep) >= -3.0f * B2_LINEAR_SLOP;
                }
                pos[ka] = ca; pos[kb] = cb;
                S.solved()[oseed] = ok;
            }
        } else if (ohead != EW_NONE) {
            const uint32_t* t_ew = S.t_ew();
            const uint32_t ew_head = t_ew[ohead];
            bool ok = false;
            for (int it = 0; it < P.pos_iters && !ok; ++it) {
                float min_sep = 0.0f;
                uint32_t ew = ew_head;
                for (;;) {
                    const int a = EWT::a(ew), b = EWT::b(ew), tn = EWT::na(ew);
                    float2 ca = pos[a], cb = pos[b];
                    uint32_t ew2 = 0u;
                    if (tn != EW_NONE) ew2 = t_ew[tn];
                    const float sep = solve_position(P.radius, P.k_sum, P.inv_mass, ca, cb);
                    pos[a] = ca; pos[b] = cb;
                    min_sep = b2min(min_sep, sep);
                    if (tn == EW_NONE) break;
                    ew = ew2;
                }
                ok = min_sep >= -3.0f * B2_LINEAR_SLOP;
            }
            S.solved()[oseed] = ok;
        }
        g.sync();
#pragma unroll
        for (int s = 0; s < APL; ++s) c[s] = pos[g.gl + s * G];
    }

    PHASE_STAMP(7);
    // ---- phase 8: sleeping (b2Island::Solve tail) --------------------------------------------------
    {
        bool cand = false;
        const float tol2 = B2_LINEAR_SLEEP_TOLERANCE * B2_LINEAR_SLEEP_TOLERANCE;
#pragma unroll
        for (int s = 0; s < APL; ++s) {
            if (!now_alive[s]) continue;
            if ((v[s].x * v[s].x + v[s].y * v[s].y) > tol2) slp[s] = 0.0f;
            else slp[s] += P.h;
            cand |= slp[s] >= B2_TIME_TO_SLEEP;
        }
        if (g.ballot(cand)) {
            uint32_t* isl_min = S.isl_min();
#pragma unroll
            for (int s = 0; s < APL; ++s) isl_min[g.gl + s * G] = 0x7f7fffffu;  // b2_maxFloat
            g.sync();
#pragma unroll
            for (int s = 0; s < APL; ++s)
                if (now_alive[s]) atomicMin(&isl_min[label[g.gl + s * G]], __float_as_uint(slp[s]));
            g.sync();
#pragma unroll
            for (int s = 0; s < APL; ++s) {
                const int isl = label[g.gl + s * G];
                const bool solved = S.solved()[isl] != 0;
                if (now_alive[s] && __uint_as_float(isl_min[isl]) >= B2_TIME_TO_SLEEP && solved) {
                    // SetAwake(false); the next ApplyForce(wake=True) wakes the body again
                    slp[s] = 0.0f; v[s] = make_float2(0.0f, 0.0f);
                }
            }
        }
    }

    PHASE_STAMP(8);
    // ---- phase 9: SynchronizeFixtures -> b2DynamicTree::MoveProxy -----------------------------------
    ASet moved = {};
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        const float r = P.radius;
        const float lox = b2min(c0[s].x - r, c[s].x - r), loy = b2min(c0[s].y - r, c[s].y - r);
        const float hix = b2max(c0[s].x + r, c[s].x + r), hiy = b2max(c0[s].y + r, c[s].y + r);
        const bool contains = fatr[s].x <= lox && fatr[s].y <= loy && hix <= fatr[s].z && hiy <= fatr[s].w;
        const bool mv = now_alive[s] && !contains;
        if (mv) {
            float nlx = lox - B2_AABB_EXTENSION, nly = loy - B2_AABB_EXTENSION;
            float nhx = hix + B2_AABB_EXTENSION, nhy = hiy + B2_AABB_EXTENSION;
            const float dx = B2_AABB_MULTIPLIER * (c[s].x - c0[s].x), dy = B2_AABB_MULTIPLIER * (c[s].y - c0[s].y);
            if (dx < 0.0f) nlx += dx; else nhx += dx;
            if (dy < 0.0f) nly += dy; else nhy += dy;
            fatr[s] = make_float4(nlx, nly, nhx, nhy);
            fat[i] = fatr[s];
        }
        const unsigned bm = g.ballot(mv);
        put_slot<G>(moved, s, bm);
    }
    g.sync();

    PHASE_STAMP(9);
    // ---- phase 10: FindNewContacts ------------------------------------------------------------------
    if (set_nonzero(moved)) cnt = find_new_contacts<G, APL>(g, S, P, moved, alive, cnt, c_ab, c_imp, overflow_c);

    PHASE_STAMP(10);
    // ---- phase 11: rewards (mvmnt.py:160-179), time/done (mvmnt.py:134-136) ---------------------------
    const int step = step_cnt + 1;
    bool done = step >= P.done_step;
    if (TDM) {
        // alive_teams (combat.py:172-182)
        int teams_alive = 0, last = -1;
        for (int t = 0; t < MACM_MAX_TEAMS; ++t) {
            bool mine = false;
#pragma unroll
            for (int s = 0; s < APL; ++s) mine |= now_alive[s] && team[s] == t;
            if (g.ballot(mine)) { ++teams_alive; last = t; }
        }
        if (teams_alive == 1) { done = true; winner = last; }
        if (teams_alive == 0) done = true;
    }
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        if (!valid[s]) continue;
        const size_t gi = (size_t)env * N + i;
        const bool col = set_nonzero(adj[i]);
        float rew = -1.0f;
        if (TDM) {
            rew = (now_alive[s] && col) ? -1.0f : 0.0f;   // SURVEY App. B12
        } else if (!col) {
            const float2 tg = S.tgt()[i];
            const float dx = tg.x - c[s].x, dy = tg.y - c[s].y;
            const float d2 = dx * dx + dy * dy;
            if (P.reward_mode == MACM_REWARD_LINEAR) rew = 1.0f - out_sqrtf(d2) * (1.0f / 35.0f);   // 1 - d/35 (mvmnt.py:179), float64 there
            else rew = (d2 < P.binary_thr) ? 1.0f : 0.0f;
        }
        if (R.rewards()) R.rewards()[(size_t)ks * EN + gi] = rew;
        if (R.collided()) R.collided()[(size_t)ks * EN + gi] = (uint8_t)col;
        if (TDM) S.ang()[i] = ang[s];
        if (!last) continue;
        P.rewards[gi] = rew;
        P.collided[gi] = (uint8_t)col;
        // ---- phase 12: write state back (last step of the launch) ----
        P.posvel[gi] = make_float4(c[s].x, c[s].y, v[s].x, v[s].y);
        P.angsleep[gi] = make_float2(ang[s], slp[s]);
        P.fat[gi] = fatr[s];
        if (TDM) P.tdm[gi] = make_float4(health[s], __int_as_float(cd_atk[s]), __int_as_float(cd_mov[s]),
                                         __int_as_float((now_alive[s] ? 1 : 0) | (hits[s] << 8)));
    }

    {
        const bool oc = g.ballot(overflow_c) != 0, ot = g.ballot(overflow_t) != 0;
        eflags = (eflags & ~MACM_ENV_FRESH) | (oc ? MACM_ENV_CONTACT_OVERFLOW : 0) | (ot ? MACM_ENV_TOUCH_OVERFLOW : 0);
        step_cnt = step;
        if (g.gl == 0) {
            if (R.done()) R.done()[(size_t)ks * P.E + env] = (uint8_t)done;
            if (last) {
                P.c_cnt[env] = cnt;
                P.done[env] = (uint8_t)done;
                P.env_state[env] = make_int4(step, eflags, tc, winner);
            }
        }
    }
    if (TDM) {
#pragma unroll
        for (int s = 0; s < APL; ++s) was_alive[s] = now_alive[s];
    }

    PHASE_STAMP(11);
    // Between two steps of a rollout the velocities, fat AABBs and sleep timers wait in shared memory (the
    // velocity array and the touching-contact stage, both idle until the next step's phase 2), so that the
    // nearest-agent search of phase 13 -- the register-hungriest phase -- does not have to carry them.
    float4* fat_park = reinterpret_cast<float4*>(S.t_n());
    float* slp_park = reinterpret_cast<float*>(fat_park + NC);
    if (ROLL && !last) {
        g.sync();
#pragma unroll
        for (int s = 0; s < APL; ++s) {
            const int i = g.gl + s * G;
            vel[i] = v[s];
            fat_park[i] = fatr[s];
            slp_park[i] = slp[s];
        }
    }
    // Auto-reset inside a rollout (MACM_FLAG_AUTO_RESET): an env that is done starts its next episode before the
    // step's observation is written -- the draws, the body creation and the order of events of macm_reset_masked
    // (the launch the flag appends to a single step), so K steps in one launch stay bit-identical to K single
    // steps.  The launch's last step leaves the reset to that appended launch: its state is already written back.
    // With final destinations given (R.finals), phase 13 first runs on the finished episode (pass 0) and stores its
    // terminal observation and state there, as macm_reset_masked copies them; then the reset and pass 1.  One copy
    // of the observation code serves both passes: code size is what limits a rollout (DESIGN, instruction supply).
    const bool restart = ROLL && !last && (P.flags & MACM_FLAG_AUTO_RESET) && done;
#pragma unroll 1
    for (int pass = (restart && R_.finals) ? 0 : 1;; ++pass) {
    if (ROLL && pass == 0) {   // terminal TDM state and env state, as phase 12 and the env-state store above write them
        if (TDM) {
#pragma unroll
            for (int s = 0; s < APL; ++s) {
                if (!valid[s]) continue;
                const size_t gi = (size_t)env * N + g.gl + s * G;
                const float4 td = make_float4(health[s], __int_as_float(cd_atk[s]), __int_as_float(cd_mov[s]),
                                              __int_as_float((now_alive[s] ? 1 : 0) | (hits[s] << 8)));
                if (R_.fin.tdm) R_.fin.tdm[gi] = td;
                if (R_.fin_k.tdm) R_.fin_k.tdm[(size_t)ks * EN + gi] = td;
            }
        }
        if (g.gl == 0) {
            const int4 es = make_int4(step_cnt, eflags, tc, winner);
            if (R_.fin.es) R_.fin.es[env] = es;
            if (R_.fin_k.es) R_.fin_k.es[(size_t)ks * P.E + env] = es;
        }
    }
    if (restart && pass == 1) {
        const uint32_t episode = ((uint32_t)eflags >> MACM_ENV_EPISODE_SHIFT) + 1u;
        g.sync();
#pragma unroll
        for (int s = 0; s < APL; ++s) {
            const int i = g.gl + s * G;
            if (valid[s]) {
                float x, y, a;
                sample_agent(P, R_.sc, (uint64_t)env * N + i + (uint64_t)P.env_base * N, i, episode, x, y, a);
                const float r = P.radius;
                c[s] = make_float2(x, y); ang[s] = a;
                vel[i] = make_float2(0.0f, 0.0f);
                fat_park[i] = make_float4((x - r) - B2_AABB_EXTENSION, (y - r) - B2_AABB_EXTENSION,
                                          (x + r) + B2_AABB_EXTENSION, (y + r) + B2_AABB_EXTENSION);
                slp_park[i] = 0.0f;
                pos[i] = c[s];
                if (TDM) { health[s] = P.init_health; cd_atk[s] = 0; cd_mov[s] = 0; hits[s] = 0; S.ang()[i] = a; }
                else S.tgt()[i] = sample_target(R_.sc, (uint64_t)(env + P.env_base) * P.T + (P.T == 1 ? 0 : (int)P.target_idx[i]), episode);
            }
            if (TDM) now_alive[s] = valid[s];
        }
        if (!TDM)
            for (int t = g.gl; t < P.T; t += G)
                const_cast<float2*>(P.targets)[(size_t)env * P.T + t] = sample_target(R_.sc, (uint64_t)(env + P.env_base) * P.T + t, episode);
        if (TDM) {
            alive = ASet{};
#pragma unroll
            for (int s = 0; s < APL; ++s) { put_slot<G>(alive, s, g.ballot(valid[s])); was_alive[s] = valid[s]; }
        }
        cnt = 0; step_cnt = 0; winner = -1;
        eflags = MACM_ENV_FRESH | (int)(episode << MACM_ENV_EPISODE_SHIFT);
        g.sync();
    }
    // ---- phase 13: observations (mvmnt.py:181-222 / combat.py:206-227) ----------------------------
    // (a rollout without per-step observation arrays only observes after its last step)
    // (pass 0 only observes when the terminal observation has somewhere to go)
    const bool obs0 = ROLL && pass == 0 &&
                      (R_.fin.obs || R_.fin_k.obs || (!TDM && (R_.fin.nn_idx || R_.fin_k.nn_idx)));
    if (((last || R.obs() || R.policy() == MACM_BOT_FLOCK) && !(ROLL && pass == 0)) || obs0) {
        float* ob_k = R.obs() ? R.obs() + (size_t)ks * EN * P.obs_words : nullptr;
        int* nn_k = R.nn_idx() ? R.nn_idx() + (size_t)ks * EN : nullptr;
        float* ob1 = last ? P.obs : ob_k;
        float* ob2 = last ? ob_k : nullptr;
        int* nn1 = last ? P.nn_idx : nn_k;
        int* nn2 = last ? nn_k : nullptr;
        // the flock actor steers by the new episode's first observation, as macm_bot_actions after the reset does
        float2* tgo = (R.policy() == MACM_BOT_FLOCK && !last) ? reinterpret_cast<float2*>(S.nw()) : nullptr;
        if (ROLL && pass == 0) {
            ob1 = R_.fin.obs;
            ob2 = R_.fin_k.obs ? R_.fin_k.obs + (size_t)ks * EN * P.obs_words : nullptr;
            nn1 = R_.fin.nn_idx;
            nn2 = R_.fin_k.nn_idx ? R_.fin_k.nn_idx + (size_t)ks * EN : nullptr;
            tgo = nullptr;
        }
        if (TDM) {
            g.sync();
            tdm_observe<G, APL>(g, S, P, env, alive, ob1, ob2);
        } else {
            flock_observe<G, APL>(g, S, P, env, ang, ob1, nn1, ob2, nn2, tgo);
        }
    }
    if (!ROLL || pass == 1) break;
    }   // for pass
    PHASE_STAMP(12);
    }   // for ks
#ifndef MACM_PHASE_TRACE
    if (P.trace && g.gl == 0) {   // macm_set_trace: per-env timing record
        unsigned long long t1, smid;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        asm volatile("{.reg .u32 t; mov.u32 t, %%smid; cvt.u64.u32 %0, t;}" : "=l"(smid));
        unsigned long long* tr = P.trace + (size_t)env * 4;
        tr[0] = tr_t0; tr[1] = t1; tr[2] = clock64() - tr_c0;
        tr[3] = smid | ((unsigned long long)tc << 16) | ((unsigned long long)nlev << 32) | ((unsigned long long)multi << 48) |
                ((unsigned long long)(slot & 0x7fff) << 49);
    }
#else
    if (P.trace && g.gl == 0) P.trace[(size_t)env * 16 + 15] = (unsigned long long)tc | ((unsigned long long)multi << 16);
#endif
}

// The group copies row `row` (n 32-bit words) of an array to the same row of up to two arrays of its layout: 16-byte
// vectors when n is a multiple of 4 and all three arrays start 16-byte aligned (every row then does too), single words
// otherwise (cartesian observations of an odd N; nn_idx arrays, which need only 4-byte alignment).
template <int G>
__device__ __forceinline__ void copy_row(const Grp<G>& g, const void* src, void* d1, void* d2, size_t row, int n)
{
    const bool vec = (n & 3) == 0 && (((uintptr_t)src | (uintptr_t)d1 | (uintptr_t)d2) & 15) == 0;   // warp-uniform
    if (vec) {
        const int n4 = n >> 2;
        const uint4* s = reinterpret_cast<const uint4*>(src) + row * n4;
        uint4* a = d1 ? reinterpret_cast<uint4*>(d1) + row * n4 : nullptr;
        uint4* b = d2 ? reinterpret_cast<uint4*>(d2) + row * n4 : nullptr;
        for (int k = g.gl; k < n4; k += G) {
            const uint4 v = s[k];
            if (a) a[k] = v;
            if (b) b[k] = v;
        }
    } else {
        const uint32_t* s = reinterpret_cast<const uint32_t*>(src) + row * n;
        uint32_t* a = d1 ? reinterpret_cast<uint32_t*>(d1) + row * n : nullptr;
        uint32_t* b = d2 ? reinterpret_cast<uint32_t*>(d2) + row * n : nullptr;
        for (int k = g.gl; k < n; k += G) {
            const uint32_t v = s[k];
            if (a) a[k] = v;
            if (b) b[k] = v;
        }
    }
}

// get_obs() alone; with RESET, first a new episode for the envs selected by `mask` (null: the bound `done`
// buffer) and nothing at all for the others -- macm_reset_masked: the reference's env.reset() (mvmnt.py:224-233,
// combat.py:229-239) for the envs that are done (mvmnt.py:134-136, combat.py:171-182).  Before anything of a
// selected env is overwritten, its rows of obs / nn_idx / tdm_state / env_state go to `fin` (the bound final slots)
// and `fin2` (row K-1 of a rollout's final_* arrays); both are unused without RESET.
template <int G, int APL, int KIND, bool RESET>
__global__ void __launch_bounds__(128) macm_observe_kernel(const __grid_constant__ SimConst P, const uint8_t* __restrict__ mask,
                                                           const __grid_constant__ SampleConst sc,
                                                           const __grid_constant__ Finals fin, const __grid_constant__ Finals fin2)
{
    constexpr int NC = G * APL;
    constexpr int GPW = 32 / G;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Grp<G> g;
    const int slot_in_block = (threadIdx.x >> 5) * GPW + (threadIdx.x & 31) / G;
    const int env = blockIdx.x * (blockDim.x / 32) * GPW + slot_in_block;
    if (env >= P.E) return;
    EnvS<NC> S;
    S.TC = P.TC;
    S.base = smem_raw + (size_t)slot_in_block * Lay<NC>::bytes(P.TC);
    if (RESET) {
        if (!(mask ? mask[env] : P.done[env])) return;   // the whole group leaves together
        if (fin.obs || fin.nn_idx || fin.tdm || fin.es || fin2.obs || fin2.nn_idx || fin2.tdm || fin2.es) {
            if (fin.obs || fin2.obs) copy_row<G>(g, P.obs, fin.obs, fin2.obs, env, P.N * P.obs_words);
            if (KIND != MACM_ENV_TDM && (fin.nn_idx || fin2.nn_idx)) copy_row<G>(g, P.nn_idx, fin.nn_idx, fin2.nn_idx, env, P.N);
            if (KIND == MACM_ENV_TDM && (fin.tdm || fin2.tdm)) copy_row<G>(g, P.tdm, fin.tdm, fin2.tdm, env, P.N * 4);
            if (fin.es || fin2.es) copy_row<G>(g, P.env_state, fin.es, fin2.es, env, 4);
            g.sync();   // every lane's loads are done before any of the rows is overwritten below
        }
        // episode counter of the env: bits 8.. of its flag word; keys the draws so that episodes differ
        const uint32_t episode = ((uint32_t)P.env_state[env].y >> MACM_ENV_EPISODE_SHIFT) + 1u;
        const float r = P.radius;
#pragma unroll
        for (int s = 0; s < APL; ++s) {
            const int i = g.gl + s * G;
            if (i >= P.N) continue;
            const size_t gi = (size_t)env * P.N + i;
            float x, y, a;
            sample_agent(P, sc, gi + (uint64_t)P.env_base * P.N, i, episode, x, y, a);
            // body creation (mvmnt.py:70-75): at rest, awake, fat AABB = tight +- b2_aabbExtension
            P.posvel[gi] = make_float4(x, y, 0.0f, 0.0f);
            P.angsleep[gi] = make_float2(a, 0.0f);
            P.fat[gi] = make_float4((x - r) - B2_AABB_EXTENSION, (y - r) - B2_AABB_EXTENSION,
                                    (x + r) + B2_AABB_EXTENSION, (y + r) + B2_AABB_EXTENSION);
            // (rewards, collided and done keep the values of the env's last step: the learner reads the terminal
            //  reward next to the new episode's first observation)
            if (KIND == MACM_ENV_TDM)
                P.tdm[gi] = make_float4(P.init_health, __int_as_float(0), __int_as_float(0), __int_as_float(1));
        }
        if (KIND != MACM_ENV_TDM)
            for (int t = g.gl; t < P.T; t += G)
                const_cast<float2*>(P.targets)[(size_t)env * P.T + t] =
                    sample_target(sc, (uint64_t)(env + P.env_base) * P.T + t, episode);
        if (g.gl == 0) {
            P.c_cnt[env] = 0;
            P.env_state[env] = make_int4(0, MACM_ENV_FRESH | (int)(episode << MACM_ENV_EPISODE_SHIFT), 0, -1);
        }
        __threadfence_block();
        g.sync();   // the group's stores (targets) are visible to its lanes below
    }
    float ang[APL];
    AgentSet<NC> alive = {};
#pragma unroll
    for (int s = 0; s < APL; ++s) {
        const int i = g.gl + s * G;
        const bool ok = i < P.N;
        const size_t gi = (size_t)env * P.N + (ok ? i : 0);
        const float4 pv = P.posvel[gi];
        ang[s] = P.angsleep[gi].x;
        S.pos()[i] = ok ? make_float2(pv.x, pv.y) : make_float2(3.0e30f, 3.0e30f);
        S.ang()[i] = ang[s];
        if (KIND != MACM_ENV_TDM) {
            const float2* tg = P.targets + (size_t)env * P.T + P.target_idx[ok ? i : 0];
            float2 tv;
            if (RESET) asm volatile("ld.volatile.global.v2.f32 {%0, %1}, [%2];" : "=f"(tv.x), "=f"(tv.y) : "l"(tg));
            else tv = *tg;
            S.tgt()[i] = tv;
        }
        bool al = ok;
        if (KIND == MACM_ENV_TDM) al = ok && (__float_as_int(P.tdm[gi].w) & 1);
        const unsigned bm = g.ballot(al);
        put_slot<G>(alive, s, bm);
    }
    g.sync();
    if (KIND == MACM_ENV_TDM) tdm_observe<G, APL>(g, S, P, env, alive, P.obs, nullptr);
    else flock_observe<G, APL>(g, S, P, env, ang, P.obs, P.nn_idx, nullptr, nullptr);
}

// Body creation for every agent (mvmnt.py:61-76): fat AABB = tight +- b2_aabbExtension, awake,
// sleep time 0, no contacts, first-step flag.  One thread per agent.
__global__ void macm_reset_kernel(const __grid_constant__ SimConst P)
{
    const size_t gi = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)P.E * P.N;
    if (gi >= total) return;
    const float4 pv = P.posvel[gi];
    const float r = P.radius;
    P.fat[gi] = make_float4((pv.x - r) - B2_AABB_EXTENSION, (pv.y - r) - B2_AABB_EXTENSION,
                            (pv.x + r) + B2_AABB_EXTENSION, (pv.y + r) + B2_AABB_EXTENSION);
    float2 as = P.angsleep[gi];
    as.y = 0.0f;
    P.angsleep[gi] = as;
    P.rewards[gi] = 0.0f;
    P.collided[gi] = 0;
    if (P.kind == MACM_ENV_TDM) P.tdm[gi] = make_float4(P.init_health, __int_as_float(0), __int_as_float(0), __int_as_float(1));
    if (gi % P.N == 0) {
        const size_t e = gi / P.N;
        P.c_cnt[e] = 0;
        P.env_state[e] = make_int4(0, MACM_ENV_FRESH, 0, -1);
        P.done[e] = 0;
    }
}

template <int G, int APL, int KIND>
cudaError_t launch_one(const SimConst& P, const LaunchCfg& cfg, const void* actions, const Rollout& R, cudaStream_t s,
                       bool observe_only)
{
#if !MACM_HUGE_BUILD
    if (observe_only) {
        macm_observe_kernel<G, APL, KIND, false><<<cfg.obs_blocks, 128, cfg.obs_smem_bytes, s>>>(P, nullptr, SampleConst{},
                                                                                                 Finals{}, Finals{});
        return cudaGetLastError();
    }
#endif
    // the step kernel is launched with programmatic stream serialization: it may become resident
    // before its predecessor in the stream has finished and waits in griddepcontrol.wait
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)cfg.blocks);
    lc.blockDim = dim3((unsigned)cfg.threads);
    lc.dynamicSmemBytes = (size_t)cfg.smem_bytes;
    lc.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = at;
    lc.numAttrs = 1;
#if MACM_HUGE_BUILD   // (two instantiations per shape: the single step and the general one)
    if (R.K == 1 && R.policy < 0 && actions && !R.obs && !R.nn_idx && !R.rewards && !R.collided && !R.done)
        return cudaLaunchKernelEx(&lc, macm_step_kernel<G, APL, KIND, 0>, P, actions, R);
    return cudaLaunchKernelEx(&lc, macm_step_kernel<G, APL, KIND, 1>, P, actions, R);
#else
    if (P.scratch != nullptr) return macm_launch_step_huge(P, cfg, actions, R, s);   // max_touching > 240: macm_kernels_huge.cu
    if (R.K == 1 && R.policy < 0 && actions) {
        if (!R.obs && !R.nn_idx && !R.rewards && !R.collided && !R.done)
            return cudaLaunchKernelEx(&lc, macm_step_kernel<G, APL, KIND, 0>, P, actions, R);
        return cudaLaunchKernelEx(&lc, macm_step_kernel<G, APL, KIND, 2>, P, actions, R);
    }
    return cudaLaunchKernelEx(&lc, macm_step_kernel<G, APL, KIND, 1>, P, actions, R);
#endif
}

#if !MACM_HUGE_BUILD
template <int G, int APL, int KIND>
cudaError_t reset_masked_one(const SimConst& P, const LaunchCfg& cfg, const uint8_t* mask, const SampleConst& sc,
                             const Finals& fin, const Finals& fin2, cudaStream_t s)
{
    macm_observe_kernel<G, APL, KIND, true><<<cfg.obs_blocks, 128, cfg.obs_smem_bytes, s>>>(P, mask, sc, fin, fin2);
    return cudaGetLastError();
}
#endif

template <int G, int APL, int KIND>
cudaError_t prepare_one(const LaunchCfg& cfg, int* blocks_per_sm)
{
    cudaError_t e = cudaFuncSetAttribute(macm_step_kernel<G, APL, KIND, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         cfg.smem_bytes);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(macm_step_kernel<G, APL, KIND, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, cfg.smem_bytes);
    if (e != cudaSuccess) return e;
#if MACM_HUGE_BUILD
    (void)blocks_per_sm;
    return cudaSuccess;
#else
    e = cudaFuncSetAttribute(macm_step_kernel<G, APL, KIND, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, cfg.smem_bytes);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(macm_observe_kernel<G, APL, KIND, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             cfg.obs_smem_bytes);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(macm_observe_kernel<G, APL, KIND, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             cfg.obs_smem_bytes);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, macm_step_kernel<G, APL, KIND, 0>, cfg.threads,
                                                         cfg.smem_bytes);
#endif
}

}  // namespace

#if !MACM_HUGE_BUILD
// lanes per env / agents per lane for a given N
static void pick_shape(int N, int* G, int* APL)
{
    if (N <= 4) { *G = 4; *APL = 1; }
    else if (N <= 8) { *G = 8; *APL = 1; }
    else if (N <= 16) { *G = 16; *APL = 1; }
    else if (N <= 32) { *G = 32; *APL = 1; }
    else if (N <= 64) { *G = 32; *APL = 2; }
    else { *G = 32; *APL = 4; }
}

cudaError_t macm_launch_cfg(const SimConst& P, int sm_count, LaunchCfg* cfg)
{
    pick_shape(P.N, &cfg->G, &cfg->APL);
    const int gpw = 32 / cfg->G;
    cfg->threads = 128;
    // one-env-per-warp groups: a block per SM (profiles/README.md, finding 4) unless the last wave of such
    // blocks would leave most SMs idle
    const int wide_threads = shape_max_threads(cfg->G, cfg->APL);
    const int wide_warps = wide_threads / 32;
    if (gpw == 1 && sm_count > 0 && P.E >= wide_warps) {
        const int wb = (P.E + wide_warps - 1) / wide_warps;
        const int waves = (wb + sm_count - 1) / sm_count;
        if (wb * 5 >= waves * sm_count * 4) cfg->threads = wide_threads;   // >= 80 % of the slots used
    }
    if (const char* e = getenv("MACM_BLOCK_THREADS")) {   // experiments (profiles/README.md): 128 or 896
        const int t = atoi(e);
        if (t == 128 || (t > 128 && t <= wide_threads && t % 32 == 0)) cfg->threads = t;
    }
    cfg->envs_per_block = (cfg->threads / 32) * gpw;
    cfg->blocks = (P.E + cfg->envs_per_block - 1) / cfg->envs_per_block;
    const int NC = cfg->G * cfg->APL;
    int per_env = 0;
    switch (NC) {
        case 4: per_env = Lay<4>::bytes(P.TC); break;
        case 8: per_env = Lay<8>::bytes(P.TC); break;
        case 16: per_env = Lay<16>::bytes(P.TC); break;
        case 32: per_env = Lay<32>::bytes(P.TC); break;
        case 64: per_env = Lay<64>::bytes(P.TC); break;
        default: per_env = Lay<128>::bytes(P.TC); break;
    }
    cfg->per_env_bytes = per_env;
    if (per_env * cfg->envs_per_block + MACM_TABLE_BYTES > 227 * 1024) {   // fall back to narrow blocks
        cfg->threads = 128;
        cfg->envs_per_block = 4 * gpw;
        cfg->blocks = (P.E + cfg->envs_per_block - 1) / cfg->envs_per_block;
    }
    cfg->smem_bytes = per_env * cfg->envs_per_block + (cfg->threads > 128 ? MACM_TABLE_BYTES : 0);   // + sin/cos table
    cfg->obs_blocks = (P.E + 4 * gpw - 1) / (4 * gpw);
    cfg->obs_smem_bytes = per_env * 4 * gpw;
    return cfg->smem_bytes <= 227 * 1024 ? cudaSuccess : cudaErrorInvalidConfiguration;
}

#endif   // !MACM_HUGE_BUILD

#define DISPATCH_SHAPE(CALL)                                                        \
    switch ((cfg.G * 8 + cfg.APL) * 2 + (P.kind == MACM_ENV_TDM ? 1 : 0)) {         \
        case (4 * 8 + 1) * 2: return CALL(4, 1, MACM_ENV_FLOCK);                    \
        case (8 * 8 + 1) * 2: return CALL(8, 1, MACM_ENV_FLOCK);                    \
        case (16 * 8 + 1) * 2: return CALL(16, 1, MACM_ENV_FLOCK);                  \
        case (32 * 8 + 1) * 2: return CALL(32, 1, MACM_ENV_FLOCK);                  \
        case (32 * 8 + 2) * 2: return CALL(32, 2, MACM_ENV_FLOCK);                  \
        case (32 * 8 + 4) * 2: return CALL(32, 4, MACM_ENV_FLOCK);                  \
        case (4 * 8 + 1) * 2 + 1: return CALL(4, 1, MACM_ENV_TDM);                  \
        case (8 * 8 + 1) * 2 + 1: return CALL(8, 1, MACM_ENV_TDM);                  \
        case (16 * 8 + 1) * 2 + 1: return CALL(16, 1, MACM_ENV_TDM);                \
        case (32 * 8 + 1) * 2 + 1: return CALL(32, 1, MACM_ENV_TDM);                \
        case (32 * 8 + 2) * 2 + 1: return CALL(32, 2, MACM_ENV_TDM);                \
        case (32 * 8 + 4) * 2 + 1: return CALL(32, 4, MACM_ENV_TDM);                \
        default: return cudaErrorInvalidConfiguration;                              \
    }

#if MACM_HUGE_BUILD
// the exports of macm_kernels_huge.cu
cudaError_t macm_prepare_kernels_huge(const SimConst& P, const LaunchCfg& cfg)
{
    int unused = 0;
#define CALL(G_, A_, K_) prepare_one<G_, A_, K_>(cfg, &unused)
    DISPATCH_SHAPE(CALL)
#undef CALL
}

cudaError_t macm_launch_step_huge(const SimConst& P, const LaunchCfg& cfg, const void* actions, const Rollout& R, cudaStream_t s)
{
#define CALL(G_, A_, K_) launch_one<G_, A_, K_>(P, cfg, actions, R, s, false)
    DISPATCH_SHAPE(CALL)
#undef CALL
}
#else
cudaError_t macm_prepare_kernels(const SimConst& P, const LaunchCfg& cfg, int* blocks_per_sm)
{
#define CALL(G_, A_, K_) prepare_one<G_, A_, K_>(cfg, blocks_per_sm)
    DISPATCH_SHAPE(CALL)
#undef CALL
}

cudaError_t macm_launch_step(const SimConst& P, const LaunchCfg& cfg, const void* actions, const Rollout& R, cudaStream_t s)
{
#define CALL(G_, A_, K_) launch_one<G_, A_, K_>(P, cfg, actions, R, s, false)
    DISPATCH_SHAPE(CALL)
#undef CALL
}

cudaError_t macm_launch_observe(const SimConst& P, const LaunchCfg& cfg, cudaStream_t s)
{
#define CALL(G_, A_, K_) launch_one<G_, A_, K_>(P, cfg, nullptr, Rollout{}, s, true)
    DISPATCH_SHAPE(CALL)
#undef CALL
}

cudaError_t macm_launch_reset_masked(const SimConst& P, const LaunchCfg& cfg, const uint8_t* mask, const SampleConst& sc,
                                     const Finals& fin, const Finals& fin2, cudaStream_t s)
{
#define CALL(G_, A_, K_) reset_masked_one<G_, A_, K_>(P, cfg, mask, sc, fin, fin2, s)
    DISPATCH_SHAPE(CALL)
#undef CALL
}

cudaError_t macm_launch_reset(const SimConst& P, cudaStream_t s)
{
    const size_t total = (size_t)P.E * P.N;
    const int threads = 256;
    macm_reset_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, s>>>(P);
    return cudaGetLastError();
}
#endif   // MACM_HUGE_BUILD
