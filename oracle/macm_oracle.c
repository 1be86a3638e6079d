/*
 * oracle/macm_oracle.c -- CPU ORACLE.  TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load this library.  The product path (gym-macm_b200/) never links, imports or calls it.
 *
 * What it is: a plain-C, scalar, deliberately literal restatement of the one hot path of
 * siyarvurucu/gym-macm -- Flock.step / TDM.step and everything they call:
 *
 *   host logic (in the reference's own float64 arithmetic)
 *     gym_macm/envs/mvmnt.py:81-140   Flock.step      (action decode, Step, rewards, time, obs)
 *     gym_macm/envs/mvmnt.py:160-179  Flock.get_rewards
 *     gym_macm/envs/mvmnt.py:181-222  Flock.get_obs
 *     gym_macm/envs/combat.py:104-184 TDM.step        (repaired semantics, SURVEY App. B)
 *     gym_macm/envs/combat.py:206-227 TDM.get_obs
 *     gym_macm/cm_framework.py:56-86  RayCastClosestCallback
 *     gym_macm/cm_framework.py:161,213-224  b2World(gravity=(0,0), doSleep=True); world.Step; ClearForces
 *     gym_macm/settings.py:25-36,110-146    constants
 *
 *   engine semantics (fp32, no FMA): the Box2D 2.3.0 subset those files exercise through
 *   pybox2d -- circle bodies, zero gravity, linear damping, stateful fat AABBs, contact
 *   lifecycle (Collide / FindNewContacts), island DFS, sequential-impulse velocity and
 *   position solvers, sleeping, closest-hit ray cast.
 *
 * PARITY UNPINNED: pybox2d is an un-vendored, un-pinned third-party dependency of the
 * reference (setup.py:5 lists only 'gym'; `from Box2D import ...` at mvmnt.py:4, combat.py:4,
 * cm_framework.py:28-33, settings.py:109).  It is not importable in the build container and
 * the reference holds no tests or golden vectors.  The engine part below is therefore a
 * restatement of upstream Box2D 2.3.0's published algorithm (b2World.cpp, b2Island.cpp,
 * b2ContactSolver.cpp, b2ContactManager.cpp, b2BroadPhase.*, b2DynamicTree.cpp, b2Body.*,
 * b2CollideCircle.cpp, b2CircleShape.cpp), kept literal on purpose: linked lists with head
 * insertion, explicit DFS stack, strictly sequential Gauss-Seidel.  It is pinned only by the
 * analytic known-answer tests of SURVEY.md Appendix D (tests/test_oracle_kat.py) and by the
 * reference's own host code executed over it (tests/golden/).
 *
 * Build: gcc -O2 -ffp-contract=off -fno-fast-math (see oracle/Makefile).  All engine math is
 * `float`; all host math is `double`, exactly where the reference's Python uses float64.
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <pthread.h>

/* ---- b2Settings.h (Box2D 2.3.0) ------------------------------------------------------- */
#define B2_PI 3.14159265359f
#define B2_EPSILON FLT_EPSILON
#define B2_MAXFLOAT FLT_MAX
#define B2_AABB_EXTENSION 0.1f
#define B2_AABB_MULTIPLIER 2.0f
#define B2_LINEAR_SLOP 0.005f
#define B2_VELOCITY_THRESHOLD 1.0f
#define B2_MAX_LINEAR_CORRECTION 0.2f
#define B2_MAX_TRANSLATION 2.0f
#define B2_MAX_TRANSLATION_SQUARED (B2_MAX_TRANSLATION * B2_MAX_TRANSLATION)
#define B2_BAUMGARTE 0.2f
#define B2_TIME_TO_SLEEP 0.5f
#define B2_LINEAR_SLEEP_TOLERANCE 0.01f

#define O_MAX_BODIES 128

typedef struct { float x, y; } V2;

static inline V2 v2(float x, float y) { V2 r; r.x = x; r.y = y; return r; }
static inline V2 v2_add(V2 a, V2 b) { return v2(a.x + b.x, a.y + b.y); }
static inline V2 v2_sub(V2 a, V2 b) { return v2(a.x - b.x, a.y - b.y); }
static inline V2 v2_scale(float s, V2 a) { return v2(s * a.x, s * a.y); }
static inline float v2_dot(V2 a, V2 b) { return a.x * b.x + a.y * b.y; }
static inline float v2_dist2(V2 a, V2 b) { V2 c = v2_sub(a, b); return v2_dot(c, c); }
static inline float v2_length(V2 a) { return sqrtf(a.x * a.x + a.y * a.y); }
static inline float b2min(float a, float b) { return a < b ? a : b; }
static inline float b2max(float a, float b) { return a > b ? a : b; }
static inline float b2clamp(float a, float lo, float hi) { return b2max(lo, b2min(a, hi)); }
/* b2Vec2::Normalize: leaves the vector unchanged when shorter than epsilon */
static inline V2 v2_normalize(V2 a)
{
    float len = v2_length(a);
    if (len < B2_EPSILON) return a;
    float inv = 1.0f / len;
    return v2(a.x * inv, a.y * inv);
}

/* ---- world ------------------------------------------------------------------------------ */
typedef struct {
    int a, b;         /* fixtureA's body (lower proxy id), fixtureB's body */
    int touching;     /* manifold.pointCount > 0 */
    int island_flag;
    float nI, tI;     /* manifold.points[0].normalImpulse / tangentImpulse */
    int prev, next;   /* world contact list (head = newest) */
    int e_prev[2], e_next[2]; /* contact edges: side 0 lives in body a's list, side 1 in body b's */
    int in_use;
} OContact;

typedef struct {
    V2 c, c0, v, f;
    float a;          /* sweep.a (fixedRotation: only SetTransform changes it) */
    float sleep_time;
    int awake, active, island_flag;
    int has_proxy;
    V2 fat_lo, fat_hi;
    int edge_head;    /* edge id = contact*2 + side, -1 = empty */
} OBody;

typedef struct {
    int n;
    OBody b[O_MAX_BODIES];
    OContact* ct;
    int ct_cap, ct_free;
    int contact_head, contact_count;
    int move_buf[O_MAX_BODIES * 2];
    int move_count;
    int new_fixture;
    float inv_dt0;
    int warm_starting;
    int damping_model; /* 0: v *= clamp(1 - h c, 0, 1) (2.3.0) ; 1: v *= 1/(1 + h c) (>= 2.3.1) */
    float radius, mass, inv_mass, friction, linear_damping;
    /* statistics of the last step */
    int last_touching, last_islands_multi;
    int last_peak_contacts;   /* most contacts the world held at once during the last step (after the prologue's
                                 FindNewContacts of a world with new fixtures, or at the end of the step) */
} OWorld;

static void ow_init(OWorld* w, int max_bodies, double radius, double density, double friction, double linear_damping,
                    int damping_model, int warm_starting)
{
    memset(w, 0, sizeof(*w));
    if (max_bodies < 2) max_bodies = 2;
    w->ct_cap = max_bodies * (max_bodies - 1) / 2;    /* every pair of the world's bodies can hold a contact */
    w->ct = (OContact*)calloc((size_t)w->ct_cap, sizeof(OContact));
    for (int i = 0; i < w->ct_cap; ++i) w->ct[i].next = i + 1;
    w->ct[w->ct_cap - 1].next = -1;
    w->ct_free = 0;
    w->contact_head = -1;
    w->radius = (float)radius;
    /* b2CircleShape::ComputeMass: mass = density * b2_pi * r * r ; b2Body::ResetMassData: invMass = 1/mass */
    w->mass = (float)density * B2_PI * w->radius * w->radius;
    w->inv_mass = 1.0f / w->mass;
    /* b2MixFriction(f1, f2) = sqrtf(f1 * f2) */
    float fr = (float)friction;
    w->friction = sqrtf(fr * fr);
    w->linear_damping = (float)linear_damping;
    w->damping_model = damping_model;
    w->warm_starting = warm_starting;
    w->inv_dt0 = 0.0f;
}

static void ow_free(OWorld* w) { free(w->ct); w->ct = NULL; }

static void ow_clear(OWorld* w)
{
    w->n = 0;
    for (int i = 0; i < w->ct_cap; ++i) { memset(&w->ct[i], 0, sizeof(OContact)); w->ct[i].next = i + 1; }
    w->ct[w->ct_cap - 1].next = -1;
    w->ct_free = 0;
    w->contact_head = -1;
    w->contact_count = 0;
    w->move_count = 0;
    w->new_fixture = 0;
    w->inv_dt0 = 0.0f;
}

static void ow_buffer_move(OWorld* w, int proxy) { w->move_buf[w->move_count++] = proxy; }

static void ow_unbuffer_move(OWorld* w, int proxy)
{
    for (int i = 0; i < w->move_count; ++i)
        if (w->move_buf[i] == proxy) w->move_buf[i] = -1;
}

/* b2World::CreateBody + b2Body::CreateFixture(circle): proxy fat AABB = tight +- 0.1, move buffered,
 * e_newFixture raised (mvmnt.py:70-75, combat.py:92-97) */
static int ow_add_body(OWorld* w, float x, float y, float angle)
{
    int i = w->n++;
    OBody* b = &w->b[i];
    memset(b, 0, sizeof(*b));
    b->c = b->c0 = v2(x, y);
    b->a = angle;
    b->awake = 1;
    b->active = 1;
    b->edge_head = -1;
    b->has_proxy = 1;
    float r = w->radius;
    b->fat_lo = v2((x - r) - B2_AABB_EXTENSION, (y - r) - B2_AABB_EXTENSION);
    b->fat_hi = v2((x + r) + B2_AABB_EXTENSION, (y + r) + B2_AABB_EXTENSION);
    ow_buffer_move(w, i);
    w->new_fixture = 1;
    return i;
}

/* b2Body::SetAwake */
static void ow_set_awake(OWorld* w, int i, int flag)
{
    OBody* b = &w->b[i];
    if (flag) {
        if (!b->awake) { b->awake = 1; b->sleep_time = 0.0f; }
    } else {
        b->awake = 0;
        b->sleep_time = 0.0f;
        b->v = v2(0.0f, 0.0f);
        b->f = v2(0.0f, 0.0f);
    }
}

/* b2Body::ApplyForce(force, point, wake=True) (mvmnt.py:118) */
static void ow_apply_force(OWorld* w, int i, float fx, float fy)
{
    OBody* b = &w->b[i];
    if (!b->awake) ow_set_awake(w, i, 1);
    if (b->awake) { b->f.x += fx; b->f.y += fy; }
}

static inline int aabb_overlap(V2 alo, V2 ahi, V2 blo, V2 bhi)
{
    /* b2TestOverlap(const b2AABB&, const b2AABB&) */
    V2 d1 = v2_sub(blo, ahi), d2 = v2_sub(alo, bhi);
    if (d1.x > 0.0f || d1.y > 0.0f) return 0;
    if (d2.x > 0.0f || d2.y > 0.0f) return 0;
    return 1;
}

static int ow_find_contact(const OWorld* w, int a, int b)
{
    /* b2ContactManager::AddPair walks bodyB's edge list looking for bodyA */
    for (int e = w->b[b].edge_head; e >= 0;) {
        const OContact* c = &w->ct[e >> 1];
        int side = e & 1;
        int other = side ? c->a : c->b;
        if (other == a) return e >> 1;
        e = c->e_next[side];
    }
    return -1;
}

static void ow_link_edge(OWorld* w, int ci, int side)
{
    OContact* c = &w->ct[ci];
    int body = side ? c->b : c->a;
    int e = ci * 2 + side;
    int head = w->b[body].edge_head;
    c->e_prev[side] = -1;
    c->e_next[side] = head;
    if (head >= 0) w->ct[head >> 1].e_prev[head & 1] = e;
    w->b[body].edge_head = e;
}

static void ow_unlink_edge(OWorld* w, int ci, int side)
{
    OContact* c = &w->ct[ci];
    int body = side ? c->b : c->a;
    int e = ci * 2 + side;
    int p = c->e_prev[side], n = c->e_next[side];
    if (p >= 0) w->ct[p >> 1].e_next[p & 1] = n;
    if (n >= 0) w->ct[n >> 1].e_prev[n & 1] = p;
    if (w->b[body].edge_head == e) w->b[body].edge_head = n;
}

/* b2ContactManager::AddPair */
static void ow_add_pair(OWorld* w, int pa, int pb)
{
    if (ow_find_contact(w, pa, pb) >= 0) return;
    int ci = w->ct_free;
    if (ci < 0) return; /* cannot happen: capacity is N(N-1)/2 */
    OContact* c = &w->ct[ci];
    w->ct_free = c->next;
    memset(c, 0, sizeof(*c));
    c->in_use = 1;
    c->a = pa; c->b = pb;
    /* insert at the head of the world list */
    c->prev = -1;
    c->next = w->contact_head;
    if (w->contact_head >= 0) w->ct[w->contact_head].prev = ci;
    w->contact_head = ci;
    ow_link_edge(w, ci, 0);
    ow_link_edge(w, ci, 1);
    ow_set_awake(w, pa, 1);
    ow_set_awake(w, pb, 1);
    ++w->contact_count;
}

/* b2ContactManager::Destroy */
static void ow_destroy_contact(OWorld* w, int ci)
{
    OContact* c = &w->ct[ci];
    if (c->prev >= 0) w->ct[c->prev].next = c->next;
    if (c->next >= 0) w->ct[c->next].prev = c->prev;
    if (w->contact_head == ci) w->contact_head = c->next;
    ow_unlink_edge(w, ci, 0);
    ow_unlink_edge(w, ci, 1);
    if (c->touching) { ow_set_awake(w, c->a, 1); ow_set_awake(w, c->b, 1); }
    c->in_use = 0;
    c->next = w->ct_free;
    w->ct_free = ci;
    --w->contact_count;
}

static int pair_less(const void* pa, const void* pb)
{
    const int* a = (const int*)pa; const int* b = (const int*)pb;
    if (a[0] != b[0]) return a[0] < b[0] ? -1 : 1;
    if (a[1] != b[1]) return a[1] < b[1] ? -1 : 1;
    return 0;
}

/* b2ContactManager::FindNewContacts -> b2BroadPhase::UpdatePairs.  The dynamic tree's query is
 * a conservative filter for exactly this fat-AABB overlap test, and the pair buffer is sorted
 * before use, so the visiting order of the tree does not matter: brute force is equivalent. */
static void ow_find_new_contacts(OWorld* w)
{
    static __thread int pairs[O_MAX_BODIES * 2 * O_MAX_BODIES][2];
    int np = 0;
    for (int i = 0; i < w->move_count; ++i) {
        int q = w->move_buf[i];
        if (q < 0) continue;
        const OBody* bq = &w->b[q];
        for (int p = 0; p < w->n; ++p) {
            if (p == q || !w->b[p].has_proxy) continue;
            if (!aabb_overlap(bq->fat_lo, bq->fat_hi, w->b[p].fat_lo, w->b[p].fat_hi)) continue;
            pairs[np][0] = p < q ? p : q;
            pairs[np][1] = p < q ? q : p;
            ++np;
        }
    }
    w->move_count = 0;
    qsort(pairs, (size_t)np, sizeof(pairs[0]), pair_less);
    int i = 0;
    while (i < np) {
        int a = pairs[i][0], b = pairs[i][1];
        ow_add_pair(w, a, b);
        ++i;
        while (i < np && pairs[i][0] == a && pairs[i][1] == b) ++i;
    }
}

/* b2Body::SetTransform(position, angle) as reached through pybox2d's `body.angle = x`
 * (mvmnt.py:103-106).  localCenter = 0, so c stays; Synchronize(xf, xf) is a no-op because the
 * fat AABB still contains the tight one; Box2D 2.3.0 then calls FindNewContacts(). */
static void ow_set_angle(OWorld* w, int i, float angle)
{
    OBody* b = &w->b[i];
    b->a = angle;
    b->c0 = b->c;
    if (b->has_proxy) {
        float r = w->radius;
        V2 lo = v2(b->c.x - r, b->c.y - r), hi = v2(b->c.x + r, b->c.y + r);
        int contains = b->fat_lo.x <= lo.x && b->fat_lo.y <= lo.y && hi.x <= b->fat_hi.x && hi.y <= b->fat_hi.y;
        if (!contains) {
            b->fat_lo = v2(lo.x - B2_AABB_EXTENSION, lo.y - B2_AABB_EXTENSION);
            b->fat_hi = v2(hi.x + B2_AABB_EXTENSION, hi.y + B2_AABB_EXTENSION);
            ow_buffer_move(w, i);
        }
    }
    ow_find_new_contacts(w);
}

/* b2Body::SetActive(false) (combat.py:162): proxies and contacts are destroyed at once */
static void ow_deactivate(OWorld* w, int i)
{
    OBody* b = &w->b[i];
    if (!b->active) return;
    b->active = 0;
    b->has_proxy = 0;
    ow_unbuffer_move(w, i);
    while (b->edge_head >= 0) ow_destroy_contact(w, b->edge_head >> 1);
}

/* b2ContactManager::Collide + b2Contact::Update + b2CollideCircles */
static void ow_collide(OWorld* w)
{
    int ci = w->contact_head;
    while (ci >= 0) {
        OContact* c = &w->ct[ci];
        const OBody* A = &w->b[c->a];
        const OBody* B = &w->b[c->b];
        if (!A->awake && !B->awake) { ci = c->next; continue; }
        if (!aabb_overlap(A->fat_lo, A->fat_hi, B->fat_lo, B->fat_hi)) {
            int nuke = ci;
            ci = c->next;
            ow_destroy_contact(w, nuke);
            continue;
        }
        int was = c->touching;
        V2 d = v2_sub(B->c, A->c);
        float dist2 = v2_dot(d, d);
        float rsum = w->radius + w->radius;
        int touching = !(dist2 > rsum * rsum);
        if (touching) {
            /* impulses survive only through a matching old manifold point (id.key 0 == 0) */
            if (!was) { c->nI = 0.0f; c->tI = 0.0f; }
        }
        c->touching = touching;
        if (touching != was) { ow_set_awake(w, c->a, 1); ow_set_awake(w, c->b, 1); }
        ci = c->next;
    }
}

typedef struct { int a, b, ci; V2 normal; float nI, tI, normal_mass, tangent_mass; } OVC;

/* b2Island::Solve for one island */
static void ow_solve_island(OWorld* w, const int* bodies, int nb, const int* contacts, int nc,
                            float h, float dt_ratio, int vel_iters, int pos_iters)
{
    static __thread V2 pc[O_MAX_BODIES], pv[O_MAX_BODIES];
    static __thread int slot[O_MAX_BODIES];
    static __thread OVC vc[O_MAX_BODIES * (O_MAX_BODIES - 1) / 2];

    /* integrate velocities and apply damping */
    for (int i = 0; i < nb; ++i) {
        OBody* b = &w->b[bodies[i]];
        slot[bodies[i]] = i;
        V2 c = b->c, v = b->v;
        b->c0 = b->c;
        /* v += h * (gravityScale * gravity + invMass * force), gravity = 0 */
        V2 acc = v2(1.0f * 0.0f + w->inv_mass * b->f.x, 1.0f * 0.0f + w->inv_mass * b->f.y);
        v.x += h * acc.x;
        v.y += h * acc.y;
        if (w->damping_model == 0)
            v = v2_scale(b2clamp(1.0f - h * w->linear_damping, 0.0f, 1.0f), v);
        else
            v = v2_scale(1.0f / (1.0f + h * w->linear_damping), v);
        pc[i] = c;
        pv[i] = v;
    }

    /* b2ContactSolver ctor + InitializeVelocityConstraints (circles, invI = 0) */
    float mA = w->inv_mass, mB = w->inv_mass;
    for (int k = 0; k < nc; ++k) {
        OContact* c = &w->ct[contacts[k]];
        OVC* q = &vc[k];
        q->ci = contacts[k];
        q->a = slot[c->a]; q->b = slot[c->b];
        if (w->warm_starting) { q->nI = dt_ratio * c->nI; q->tI = dt_ratio * c->tI; }
        else { q->nI = 0.0f; q->tI = 0.0f; }
        V2 pA = pc[q->a], pB = pc[q->b];
        V2 normal = v2(1.0f, 0.0f);
        if (v2_dist2(pA, pB) > B2_EPSILON * B2_EPSILON) normal = v2_normalize(v2_sub(pB, pA));
        q->normal = normal;
        float k_normal = mA + mB;
        q->normal_mass = k_normal > 0.0f ? 1.0f / k_normal : 0.0f;
        float k_tangent = mA + mB;
        q->tangent_mass = k_tangent > 0.0f ? 1.0f / k_tangent : 0.0f;
    }
    /* WarmStart */
    for (int k = 0; k < nc; ++k) {
        OVC* q = &vc[k];
        V2 tangent = v2(1.0f * q->normal.y, -1.0f * q->normal.x);
        V2 P = v2_add(v2_scale(q->nI, q->normal), v2_scale(q->tI, tangent));
        pv[q->a] = v2_sub(pv[q->a], v2_scale(mA, P));
        pv[q->b] = v2_add(pv[q->b], v2_scale(mB, P));
    }
    /* SolveVelocityConstraints */
    for (int it = 0; it < vel_iters; ++it) {
        for (int k = 0; k < nc; ++k) {
            OVC* q = &vc[k];
            V2 vA = pv[q->a], vB = pv[q->b];
            V2 normal = q->normal;
            V2 tangent = v2(1.0f * normal.y, -1.0f * normal.x);
            float friction = w->friction;
            {   /* tangent constraint first */
                V2 dv = v2_sub(vB, vA);
                float vt = v2_dot(dv, tangent) - 0.0f;
                float lambda = q->tangent_mass * (-vt);
                float max_friction = friction * q->nI;
                float new_impulse = b2clamp(q->tI + lambda, -max_friction, max_friction);
                lambda = new_impulse - q->tI;
                q->tI = new_impulse;
                V2 P = v2_scale(lambda, tangent);
                vA = v2_sub(vA, v2_scale(mA, P));
                vB = v2_add(vB, v2_scale(mB, P));
            }
            {   /* normal constraint */
                V2 dv = v2_sub(vB, vA);
                float vn = v2_dot(dv, normal);
                float lambda = -q->normal_mass * (vn - 0.0f);
                float new_impulse = b2max(q->nI + lambda, 0.0f);
                lambda = new_impulse - q->nI;
                q->nI = new_impulse;
                V2 P = v2_scale(lambda, normal);
                vA = v2_sub(vA, v2_scale(mA, P));
                vB = v2_add(vB, v2_scale(mB, P));
            }
            pv[q->a] = vA;
            pv[q->b] = vB;
        }
    }
    /* StoreImpulses */
    for (int k = 0; k < nc; ++k) { w->ct[vc[k].ci].nI = vc[k].nI; w->ct[vc[k].ci].tI = vc[k].tI; }

    /* integrate positions */
    for (int i = 0; i < nb; ++i) {
        V2 c = pc[i], v = pv[i];
        V2 tr = v2_scale(h, v);
        if (v2_dot(tr, tr) > B2_MAX_TRANSLATION_SQUARED) {
            float ratio = B2_MAX_TRANSLATION / v2_length(tr);
            v = v2_scale(ratio, v);
        }
        c.x += h * v.x;
        c.y += h * v.y;
        pc[i] = c;
        pv[i] = v;
    }

    /* SolvePositionConstraints */
    int position_solved = 0;
    float rA = w->radius, rB = w->radius;
    for (int it = 0; it < pos_iters; ++it) {
        float min_sep = 0.0f;
        for (int k = 0; k < nc; ++k) {
            OVC* q = &vc[k];
            V2 cA = pc[q->a], cB = pc[q->b];
            V2 normal = v2_normalize(v2_sub(cB, cA));
            float separation = v2_dot(v2_sub(cB, cA), normal) - rA - rB;
            min_sep = b2min(min_sep, separation);
            float C = b2clamp(B2_BAUMGARTE * (separation + B2_LINEAR_SLOP), -B2_MAX_LINEAR_CORRECTION, 0.0f);
            float K = mA + mB;
            float impulse = K > 0.0f ? -C / K : 0.0f;
            V2 P = v2_scale(impulse, normal);
            cA = v2_sub(cA, v2_scale(mA, P));
            cB = v2_add(cB, v2_scale(mB, P));
            pc[q->a] = cA;
            pc[q->b] = cB;
        }
        if (min_sep >= -3.0f * B2_LINEAR_SLOP) { position_solved = 1; break; }
    }

    for (int i = 0; i < nb; ++i) {
        OBody* b = &w->b[bodies[i]];
        b->c = pc[i];
        b->v = pv[i];
    }

    /* sleeping (m_allowSleep, doSleep=True at cm_framework.py:161) */
    float min_sleep = B2_MAXFLOAT;
    const float lin_tol2 = B2_LINEAR_SLEEP_TOLERANCE * B2_LINEAR_SLEEP_TOLERANCE;
    for (int i = 0; i < nb; ++i) {
        OBody* b = &w->b[bodies[i]];
        if (v2_dot(b->v, b->v) > lin_tol2) {
            b->sleep_time = 0.0f;
            min_sleep = 0.0f;
        } else {
            b->sleep_time += h;
            min_sleep = b2min(min_sleep, b->sleep_time);
        }
    }
    if (min_sleep >= B2_TIME_TO_SLEEP && position_solved)
        for (int i = 0; i < nb; ++i) ow_set_awake(w, bodies[i], 0);
}

/* b2World::Solve */
static void ow_solve(OWorld* w, float h, float dt_ratio, int vel_iters, int pos_iters)
{
    static __thread int stack[O_MAX_BODIES], ib[O_MAX_BODIES];
    static __thread int ic[O_MAX_BODIES * (O_MAX_BODIES - 1) / 2];
    for (int i = 0; i < w->n; ++i) w->b[i].island_flag = 0;
    for (int ci = w->contact_head; ci >= 0; ci = w->ct[ci].next) w->ct[ci].island_flag = 0;
    w->last_islands_multi = 0;

    /* m_bodyList is head-inserted: last created body first */
    for (int seed = w->n - 1; seed >= 0; --seed) {
        OBody* s = &w->b[seed];
        if (s->island_flag) continue;
        if (!s->awake || !s->active) continue;
        int nb = 0, nc = 0, sp = 0;
        stack[sp++] = seed;
        s->island_flag = 1;
        while (sp > 0) {
            int bi = stack[--sp];
            OBody* b = &w->b[bi];
            ib[nb++] = bi;
            ow_set_awake(w, bi, 1);
            for (int e = b->edge_head; e >= 0;) {
                OContact* c = &w->ct[e >> 1];
                int side = e & 1;
                int next = c->e_next[side];
                if (!c->island_flag && c->touching) {
                    ic[nc++] = e >> 1;
                    c->island_flag = 1;
                    int other = side ? c->a : c->b;
                    if (!w->b[other].island_flag) {
                        stack[sp++] = other;
                        w->b[other].island_flag = 1;
                    }
                }
                e = next;
            }
        }
        if (nc > 0) ++w->last_islands_multi;
        ow_solve_island(w, ib, nb, ic, nc, h, dt_ratio, vel_iters, pos_iters);
    }

    /* SynchronizeFixtures -> b2Fixture::Synchronize -> b2BroadPhase::MoveProxy -> b2DynamicTree::MoveProxy */
    for (int i = w->n - 1; i >= 0; --i) {
        OBody* b = &w->b[i];
        if (!b->island_flag) continue;
        float r = w->radius;
        V2 lo1 = v2(b->c0.x - r, b->c0.y - r), hi1 = v2(b->c0.x + r, b->c0.y + r);
        V2 lo2 = v2(b->c.x - r, b->c.y - r), hi2 = v2(b->c.x + r, b->c.y + r);
        V2 lo = v2(b2min(lo1.x, lo2.x), b2min(lo1.y, lo2.y));
        V2 hi = v2(b2max(hi1.x, hi2.x), b2max(hi1.y, hi2.y));
        V2 disp = v2_sub(b->c, b->c0);
        int contains = b->fat_lo.x <= lo.x && b->fat_lo.y <= lo.y && hi.x <= b->fat_hi.x && hi.y <= b->fat_hi.y;
        if (contains) continue;
        lo = v2(lo.x - B2_AABB_EXTENSION, lo.y - B2_AABB_EXTENSION);
        hi = v2(hi.x + B2_AABB_EXTENSION, hi.y + B2_AABB_EXTENSION);
        V2 d = v2_scale(B2_AABB_MULTIPLIER, disp);
        if (d.x < 0.0f) lo.x += d.x; else hi.x += d.x;
        if (d.y < 0.0f) lo.y += d.y; else hi.y += d.y;
        b->fat_lo = lo;
        b->fat_hi = hi;
        ow_buffer_move(w, i);
    }
    ow_find_new_contacts(w);
}

/* b2World::Step(dt, velocityIterations, positionIterations) + ClearForces (cm_framework.py:222-224) */
static void ow_step(OWorld* w, float dt, int vel_iters, int pos_iters)
{
    if (w->new_fixture) { ow_find_new_contacts(w); w->new_fixture = 0; }
    int peak = w->contact_count;
    float inv_dt = dt > 0.0f ? 1.0f / dt : 0.0f;
    float dt_ratio = w->inv_dt0 * dt;
    ow_collide(w);
    int nt = 0;
    for (int ci = w->contact_head; ci >= 0; ci = w->ct[ci].next) nt += w->ct[ci].touching;
    w->last_touching = nt;
    if (dt > 0.0f) ow_solve(w, dt, dt_ratio, vel_iters, pos_iters);
    /* SolveTOI: every contact is skipped (two non-bullet dynamic bodies) */
    if (dt > 0.0f) w->inv_dt0 = inv_dt;
    w->last_peak_contacts = peak > w->contact_count ? peak : w->contact_count;
    for (int i = 0; i < w->n; ++i) w->b[i].f = v2(0.0f, 0.0f);
}

/* b2World::RayCast with the closest-hit callback of cm_framework.py:56-86: the callback
 * returns `fraction`, which clips the ray, so the last fixture reported is the one with the
 * smallest fraction.  Exact test: b2CircleShape::RayCast against maxFraction = 1.  Which of two
 * EQUAL fractions Box2D reports last depends on its tree layout; here: lowest body index. */
static int ow_raycast_closest(const OWorld* w, V2 p1, V2 p2, float* out_fraction)
{
    int hit = -1;
    float best = 0.0f;
    for (int i = 0; i < w->n; ++i) {
        const OBody* b = &w->b[i];
        if (!b->has_proxy) continue;
        V2 s = v2_sub(p1, b->c);
        float bb = v2_dot(s, s) - w->radius * w->radius;
        V2 r = v2_sub(p2, p1);
        float c = v2_dot(s, r);
        float rr = v2_dot(r, r);
        float sigma = c * c - rr * bb;
        if (sigma < 0.0f || rr < B2_EPSILON) continue;
        float a = -(c + sqrtf(sigma));
        if (0.0f <= a && a <= 1.0f * rr) {
            a /= rr;
            if (hit < 0 || a < best) { hit = i; best = a; }
        }
    }
    if (out_fraction) *out_fraction = hit >= 0 ? best : 1.0f;
    return hit;
}

/* ---- environments (host logic of mvmnt.py / combat.py, float64 where Python is) ---------- */
typedef struct {
    int env_kind;            /* 0 flock, 1 tdm */
    int n_agents, n_targets;
    double hz;
    int velocity_iterations, position_iterations;
    double radius, density, friction, linear_damping;
    double agent_force, agent_rotation_speed;
    double time_limit;
    int reward_mode;         /* 0 binary, 1 linear */
    int action_mode;         /* 0 discrete, 1 continuous */
    int coord;               /* 0 polar, 1 cartesian */
    double reward_radius;
    int damping_model;
    int warm_starting;
    int flags;               /* bit0: repair cooldown_mov decrement (B10) */
    double cooldown_atk, cooldown_mov_penalty, melee_range, melee_dmg, percent_mov_penalty, init_health;
} OParams;

typedef struct {
    OWorld w;
    V2 targets[16];
    uint8_t target_idx[O_MAX_BODIES];
    double time_passed;
    int done, winner;
    int step_count;
    /* tdm */
    double health[O_MAX_BODIES], cd_atk[O_MAX_BODIES], cd_mov[O_MAX_BODIES];
    int alive[O_MAX_BODIES], team[O_MAX_BODIES];
} OEnv;

typedef struct {
    OParams p;
    int n_envs;
    OEnv* e;
} OBatch;

#define NP_PI 3.141592653589793

OBatch* oracle_create(const OParams* p, int n_envs)
{
    if (p->n_agents < 1 || p->n_agents > O_MAX_BODIES || p->n_targets > 16) return NULL;
    OBatch* B = (OBatch*)calloc(1, sizeof(OBatch));
    B->p = *p;
    B->n_envs = n_envs;
    B->e = (OEnv*)calloc((size_t)n_envs, sizeof(OEnv));
    for (int i = 0; i < n_envs; ++i)
        ow_init(&B->e[i].w, p->n_agents, p->radius, p->density, p->friction, p->linear_damping, p->damping_model,
                p->warm_starting);
    return B;
}

void oracle_destroy(OBatch* B)
{
    if (!B) return;
    for (int i = 0; i < B->n_envs; ++i) ow_free(&B->e[i].w);
    free(B->e);
    free(B);
}

/* Fresh worlds, as Flock.__init__ / TDM.__init__ build them (mvmnt.py:61-76, combat.py:82-98):
 * pos/angle are float64 on the Python side and become float32 at the SWIG boundary. */
static void reset_env(OBatch* B, int ei, const double* pos /*[N,2]*/, const double* angle /*[N]*/,
                      const double* targets /*[T,2] or NULL*/, const uint8_t* target_idx /*[N] or NULL*/,
                      const uint8_t* team /*[N] or NULL*/)
{
    int N = B->p.n_agents, T = B->p.n_targets;
    OEnv* e = &B->e[ei];
    ow_clear(&e->w);
    for (int i = 0; i < N; ++i) {
        ow_add_body(&e->w, (float)pos[i * 2], (float)pos[i * 2 + 1], (float)angle[i]);
        if (target_idx) e->target_idx[i] = target_idx[i];
        e->health[i] = B->p.init_health;
        e->cd_atk[i] = 0.0;
        e->cd_mov[i] = 0.0;
        e->alive[i] = 1;
        if (team) e->team[i] = team[i];
    }
    for (int t = 0; t < T; ++t)
        if (targets) e->targets[t] = v2((float)targets[t * 2], (float)targets[t * 2 + 1]);
    e->time_passed = 0.0;
    e->done = 0;
    e->winner = -1;
    e->step_count = 0;
}

void oracle_reset(OBatch* B, const double* pos /*[E,N,2]*/, const double* angle /*[E,N]*/,
                  const double* targets /*[E,T,2] or NULL*/, const uint8_t* target_idx /*[N] or NULL*/,
                  const uint8_t* team /*[N] or NULL*/)
{
    int N = B->p.n_agents, T = B->p.n_targets;
    static const uint8_t zeros[O_MAX_BODIES] = {0};
    for (int ei = 0; ei < B->n_envs; ++ei) {
        if (!targets)
            for (int t = 0; t < T; ++t) B->e[ei].targets[t] = v2(0.0f, 0.0f);
        reset_env(B, ei, pos + (size_t)ei * N * 2, angle + (size_t)ei * N, targets ? targets + (size_t)ei * T * 2 : NULL,
                  target_idx ? target_idx : zeros, team ? team : zeros);
    }
}

/* A new episode for ONE env of the batch (the reference's env.reset(), mvmnt.py:224-233 / combat.py:229-239,
 * with the repaired semantics of SURVEY App. B3: a fresh world with newly drawn bodies); target indices and
 * teams are kept. */
void oracle_reset_env(OBatch* B, int ei, const double* pos /*[N,2]*/, const double* angle /*[N]*/,
                      const double* targets /*[T,2] or NULL = keep*/)
{
    reset_env(B, ei, pos, angle, targets, NULL, NULL);
}

static inline double wrap_pi(double t)
{
    /* t - sign(t)*2*pi if |t| > pi else t   (mvmnt.py:199) */
    if (fabs(t) > NP_PI) {
        double s = (t > 0.0) - (t < 0.0);
        return t - s * 2 * NP_PI;
    }
    return t;
}

/* rotation + wrap + force of mvmnt.py:103-118 / combat.py:126-139 */
static void env_discrete_motion(OEnv* e, int i, const int* act, double rot_speed, double hz, double force)
{
    OWorld* w = &e->w;
    double ang = (double)w->b[i].a;
    double na = ang + (double)(act[2] - 1) * rot_speed * (1 / hz);
    ow_set_angle(w, i, (float)na);
    if (fabs((double)w->b[i].a) > NP_PI) {
        double a = (double)w->b[i].a;
        double s = (a > 0.0) - (a < 0.0);
        ow_set_angle(w, i, (float)(a - s * (2 * NP_PI)));
    }
    double angle = (double)w->b[i].a;
    double c = (act[0] != 1 && act[1] != 1) ? 1 / sqrt(2.0) : 1.0;
    double xf = (cos(angle) * (act[0] - 1) + cos(angle + NP_PI / 2) * (act[1] - 1)) * c * force;
    double yf = (sin(angle) * (act[0] - 1) + sin(angle + NP_PI / 2) * (act[1] - 1)) * c * force;
    ow_apply_force(w, i, (float)xf, (float)yf);
}

static void flock_observe(const OBatch* B, const OEnv* e, int32_t* nn_idx, double* nn_pos, double* tg_pos)
{
    int N = B->p.n_agents;
    const OWorld* w = &e->w;
    for (int i = 0; i < N; ++i) {
        double closest = INFINITY;
        int ca = -1;
        for (int j = 0; j < N; ++j) {
            if (j == i) continue;
            double r = sqrt((double)v2_dist2(w->b[j].c, w->b[i].c));
            if (r < closest) { ca = j; closest = r; }
        }
        nn_idx[i] = ca;
        if (ca >= 0) {
            V2 rel = v2_sub(w->b[ca].c, w->b[i].c);
            double t = wrap_pi(atan2((double)rel.y, (double)rel.x) - (double)w->b[i].a);
            nn_pos[i * 3 + 0] = closest;
            if (B->p.coord == 0) { nn_pos[i * 3 + 1] = t; nn_pos[i * 3 + 2] = 0.0; }
            else { nn_pos[i * 3 + 1] = cos(t); nn_pos[i * 3 + 2] = sin(t); }
        } else {
            nn_pos[i * 3 + 0] = INFINITY; nn_pos[i * 3 + 1] = 0.0; nn_pos[i * 3 + 2] = 0.0;
        }
        V2 tg = e->targets[e->target_idx[i]];
        V2 rel = v2_sub(tg, w->b[i].c);
        double r = sqrt((double)v2_dist2(tg, w->b[i].c));
        double t = wrap_pi(atan2((double)rel.y, (double)rel.x) - (double)w->b[i].a);
        tg_pos[i * 3 + 0] = r;
        if (B->p.coord == 0) { tg_pos[i * 3 + 1] = t; tg_pos[i * 3 + 2] = 0.0; }
        else { tg_pos[i * 3 + 1] = cos(t); tg_pos[i * 3 + 2] = sin(t); }
    }
}

static void collided_flags(const OWorld* w, uint8_t* flags, int N)
{
    /* `for contact in world.contacts` -- every listed contact, touching or not (mvmnt.py:162-164) */
    memset(flags, 0, (size_t)N);
    for (int ci = w->contact_head; ci >= 0; ci = w->ct[ci].next) {
        flags[w->ct[ci].a] = 1;
        flags[w->ct[ci].b] = 1;
    }
}

static void flock_step_env(const OBatch* B, OEnv* e, const int32_t* act_d, const double* act_c,
                           int32_t* nn_idx, double* nn_pos, double* tg_pos, double* rewards, uint8_t* collided)
{
    const OParams* p = &B->p;
    int N = p->n_agents;
    OWorld* w = &e->w;
    if (p->action_mode == 0) {
        for (int i = 0; i < N; ++i) {
            int a[3] = { act_d[i * 3], act_d[i * 3 + 1], act_d[i * 3 + 2] };
            env_discrete_motion(e, i, a, p->agent_rotation_speed, p->hz, p->agent_force);
        }
    } else {
        for (int i = 0; i < N; ++i) {
            double x = act_c[i * 2], y = act_c[i * 2 + 1];
            if ((x * x + y * y) > 1) {
                /* bug-compatible with mvmnt.py:124-126: x loses its sign, y uses the NEW x */
                x = sqrt(x * x / (x * x + y * y));
                y = sqrt(y * y / (x * x + y * y));
            }
            ow_apply_force(w, i, (float)(x * p->agent_force), (float)(y * p->agent_force));
        }
    }
    ow_step(w, (float)(1.0 / p->hz), p->velocity_iterations, p->position_iterations);

    collided_flags(w, collided, N);
    for (int i = 0; i < N; ++i) {
        if (collided[i]) { rewards[i] = -1.0; continue; }
        double d = sqrt((double)v2_dist2(e->targets[e->target_idx[i]], w->b[i].c));
        if (p->reward_mode == 1) rewards[i] = (-d / 35) + 1;
        else rewards[i] = (double)(int)(d < p->reward_radius);
    }
    e->time_passed += (1 / p->hz);
    if (e->time_passed > p->time_limit) e->done = 1;
    ++e->step_count;
    flock_observe(B, e, nn_idx, nn_pos, tg_pos);
}

static void tdm_observe(const OBatch* B, const OEnv* e, double* obs /*[N,N,3]*/, int8_t* type /*[N,N]*/)
{
    int N = B->p.n_agents;
    const OWorld* w = &e->w;
    for (int i = 0; i < N; ++i)
        for (int j = 0; j < N; ++j) {
            double* o = obs + ((size_t)i * N + j) * 3;
            if (!e->alive[i] || !e->alive[j] || i == j) {
                o[0] = o[1] = o[2] = 0.0;
                type[i * N + j] = -1;
                continue;
            }
            V2 rel = v2_sub(w->b[j].c, w->b[i].c);
            o[0] = sqrt((double)v2_dist2(w->b[j].c, w->b[i].c));
            o[1] = wrap_pi(atan2((double)rel.y, (double)rel.x) - (double)w->b[i].a);
            o[2] = wrap_pi((double)w->b[j].a - (double)w->b[i].a);
            type[i * N + j] = (int8_t)(e->team[i] == e->team[j]);
        }
}

static void tdm_step_env(const OBatch* B, OEnv* e, const int32_t* act /*[N,4]*/, double* obs, int8_t* type,
                         double* rewards, uint8_t* collided)
{
    const OParams* p = &B->p;
    int N = p->n_agents;
    OWorld* w = &e->w;
    for (int i = 0; i < N; ++i) {
        if (!e->alive[i]) continue;
        int a[3] = { act[i * 4], act[i * 4 + 1], act[i * 4 + 2] };
        /* Agent.force property (combat.py:46-49) */
        double force = p->agent_force * (1 - p->percent_mov_penalty * (int)(e->cd_mov[i] > 0));
        env_discrete_motion(e, i, a, p->agent_rotation_speed, p->hz, force);
        int attacked = 0;
        if (e->cd_atk[i] <= 0) {
            if (act[i * 4 + 3]) {
                V2 p1 = w->b[i].c;
                double ang = (double)w->b[i].a;
                V2 d = v2((float)(p->melee_range * cos(ang)), (float)(p->melee_range * sin(ang)));
                V2 p2 = v2_add(p1, d);
                int hit = ow_raycast_closest(w, p1, p2, NULL);
                e->cd_atk[i] = p->cooldown_atk;
                e->cd_mov[i] = p->cooldown_mov_penalty;
                attacked = 1;
                if (hit >= 0) e->health[hit] -= p->melee_dmg; /* B9 repaired: hit is per cast */
            }
        } else {
            e->cd_atk[i] -= (1 / p->hz);
        }
        /* B10 repaired: the movement penalty runs out like the attack cool-down does */
        if ((p->flags & 1) && !attacked && e->cd_mov[i] > 0) e->cd_mov[i] -= (1 / p->hz);
    }
    int n_alive[8] = { 0 };
    for (int i = 0; i < N; ++i) {
        if (!e->alive[i]) continue;
        if (e->health[i] <= 0) { e->alive[i] = 0; ow_deactivate(w, i); }
    }
    ow_step(w, (float)(1.0 / p->hz), p->velocity_iterations, p->position_iterations);
    tdm_observe(B, e, obs, type);
    /* B12 extension: Flock's collision penalty, 0 otherwise; dead agents get 0 */
    collided_flags(w, collided, N);
    for (int i = 0; i < N; ++i) rewards[i] = (e->alive[i] && collided[i]) ? -1.0 : 0.0;
    e->time_passed += (1 / p->hz);
    ++e->step_count;
    for (int i = 0; i < N; ++i) if (e->alive[i]) ++n_alive[e->team[i] & 7];
    int alive_teams = 0, last = -1;
    for (int t = 0; t < 8; ++t) if (n_alive[t]) { ++alive_teams; last = t; }
    if (e->time_passed > p->time_limit) e->done = 1;
    if (alive_teams == 1) { e->done = 1; e->winner = last; }
    if (alive_teams == 0) e->done = 1;
}

/* One env.step for every env of the batch. Flock outputs: nn_idx [E,N], nn_pos/tg_pos [E,N,3]
 * (polar fills 2), rewards [E,N], collided [E,N], done [E].  actions: int32 [E,N,3] or f64 [E,N,2]. */
typedef struct {
    OBatch* B; int lo, hi;
    const int32_t* act_d; const double* act_c; int32_t* nn_idx; double* nn_pos; double* tg_pos;
    double* rewards; uint8_t* collided; uint8_t* done;
    double* tobs; int8_t* ttype; int32_t* winner;
} OJob;

static void* flock_job(void* arg)
{
    OJob* j = (OJob*)arg;
    OBatch* B = j->B;
    int N = B->p.n_agents;
    for (int ei = j->lo; ei < j->hi; ++ei) {
        size_t o = (size_t)ei * N;
        flock_step_env(B, &B->e[ei], j->act_d ? j->act_d + o * 3 : NULL, j->act_c ? j->act_c + o * 2 : NULL,
                       j->nn_idx + o, j->nn_pos + o * 3, j->tg_pos + o * 3, j->rewards + o, j->collided + o);
        j->done[ei] = (uint8_t)B->e[ei].done;
    }
    return NULL;
}

/* static partition of the env range over n_threads pthreads (envs are independent) */
static void run_jobs(void* (*fn)(void*), OJob proto, int n_envs, int n_threads)
{
    if (n_threads < 1) n_threads = 1;
    if (n_threads > n_envs) n_threads = n_envs > 0 ? n_envs : 1;
    if (n_threads == 1) { proto.lo = 0; proto.hi = n_envs; fn(&proto); return; }
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)n_threads);
    OJob* jobs = (OJob*)malloc(sizeof(OJob) * (size_t)n_threads);
    for (int t = 0; t < n_threads; ++t) {
        jobs[t] = proto;
        jobs[t].lo = (int)((long long)n_envs * t / n_threads);
        jobs[t].hi = (int)((long long)n_envs * (t + 1) / n_threads);
        pthread_create(&th[t], NULL, fn, &jobs[t]);
    }
    for (int t = 0; t < n_threads; ++t) pthread_join(th[t], NULL);
    free(th);
    free(jobs);
}

void oracle_flock_step(OBatch* B, const int32_t* act_d, const double* act_c, int32_t* nn_idx, double* nn_pos,
                       double* tg_pos, double* rewards, uint8_t* collided, uint8_t* done, int n_threads)
{
    OJob j;
    memset(&j, 0, sizeof(j));
    j.B = B; j.act_d = act_d; j.act_c = act_c; j.nn_idx = nn_idx; j.nn_pos = nn_pos; j.tg_pos = tg_pos;
    j.rewards = rewards; j.collided = collided; j.done = done;
    run_jobs(flock_job, j, B->n_envs, n_threads);
}

void oracle_flock_observe(OBatch* B, int32_t* nn_idx, double* nn_pos, double* tg_pos)
{
    int N = B->p.n_agents;
    for (int ei = 0; ei < B->n_envs; ++ei) {
        size_t o = (size_t)ei * N;
        flock_observe(B, &B->e[ei], nn_idx + o, nn_pos + o * 3, tg_pos + o * 3);
    }
}

static void* tdm_job(void* arg)
{
    OJob* j = (OJob*)arg;
    OBatch* B = j->B;
    int N = B->p.n_agents;
    for (int ei = j->lo; ei < j->hi; ++ei) {
        size_t o = (size_t)ei * N;
        tdm_step_env(B, &B->e[ei], j->act_d + o * 4, j->tobs + o * N * 3, j->ttype + o * N, j->rewards + o,
                     j->collided + o);
        j->done[ei] = (uint8_t)B->e[ei].done;
        j->winner[ei] = B->e[ei].winner;
    }
    return NULL;
}

void oracle_tdm_step(OBatch* B, const int32_t* act, double* obs, int8_t* type, double* rewards, uint8_t* collided,
                     uint8_t* done, int32_t* winner, int n_threads)
{
    OJob j;
    memset(&j, 0, sizeof(j));
    j.B = B; j.act_d = act; j.tobs = obs; j.ttype = type; j.rewards = rewards; j.collided = collided;
    j.done = done; j.winner = winner;
    run_jobs(tdm_job, j, B->n_envs, n_threads);
}

void oracle_tdm_observe(OBatch* B, double* obs, int8_t* type)
{
    int N = B->p.n_agents;
    for (int ei = 0; ei < B->n_envs; ++ei) {
        size_t o = (size_t)ei * N;
        tdm_observe(B, &B->e[ei], obs + o * N * 3, type + o * N);
    }
}

/* ---- state access (parity harness) ------------------------------------------------------- */
/* body: [E,N,10] = x y vx vy angle sleep_time fat_lo.x fat_lo.y fat_hi.x fat_hi.y */
void oracle_get_bodies(const OBatch* B, float* body)
{
    int N = B->p.n_agents;
    for (int ei = 0; ei < B->n_envs; ++ei)
        for (int i = 0; i < N; ++i) {
            const OBody* b = &B->e[ei].w.b[i];
            float* o = body + ((size_t)ei * N + i) * 10;
            o[0] = b->c.x; o[1] = b->c.y; o[2] = b->v.x; o[3] = b->v.y; o[4] = b->a; o[5] = b->sleep_time;
            o[6] = b->fat_lo.x; o[7] = b->fat_lo.y; o[8] = b->fat_hi.x; o[9] = b->fat_hi.y;
        }
}

/* Contacts of env `ei` in BIRTH order (oldest first == reverse world-list order).
 * ab: [cap,2]; flags: [cap] (bit0 touching); imp: [cap,2].  Returns the count. */
int oracle_get_contacts(const OBatch* B, int ei, int32_t* ab, uint8_t* flags, float* imp, int cap)
{
    const OWorld* w = &B->e[ei].w;
    int n = w->contact_count, k = n;
    for (int ci = w->contact_head; ci >= 0; ci = w->ct[ci].next) {
        --k;
        if (k < cap && k >= 0) {
            ab[k * 2] = w->ct[ci].a; ab[k * 2 + 1] = w->ct[ci].b;
            flags[k] = (uint8_t)w->ct[ci].touching;
            imp[k * 2] = w->ct[ci].nI; imp[k * 2 + 1] = w->ct[ci].tI;
        }
    }
    return n;
}

/* Overwrite the dynamic state of env `ei` (mid-trajectory load).  Contacts are given in birth
 * order; re-inserting them oldest-first rebuilds the world list and both edge lists exactly,
 * because all three are head-inserted and removals keep relative order. */
void oracle_set_env_state(OBatch* B, int ei, const float* body /*[N,10]*/, int n_contacts, const int32_t* ab,
                          const uint8_t* flags, const float* imp, float inv_dt0, int step_count, double time_passed,
                          int new_fixture)
{
    OEnv* e = &B->e[ei];
    OWorld* w = &e->w;
    int N = B->p.n_agents;
    while (w->contact_head >= 0) ow_destroy_contact(w, w->contact_head);
    w->move_count = 0;
    for (int i = 0; i < N; ++i) {
        OBody* b = &w->b[i];
        const float* o = body + (size_t)i * 10;
        b->c = b->c0 = v2(o[0], o[1]);
        b->v = v2(o[2], o[3]);
        b->a = o[4];
        b->sleep_time = o[5];
        b->fat_lo = v2(o[6], o[7]);
        b->fat_hi = v2(o[8], o[9]);
        b->f = v2(0.0f, 0.0f);
        b->awake = 1;
        if (new_fixture && b->has_proxy) ow_buffer_move(w, i);
    }
    for (int k = 0; k < n_contacts; ++k) {
        ow_add_pair(w, ab[k * 2], ab[k * 2 + 1]);
        OContact* c = &w->ct[w->contact_head];
        c->touching = flags[k] & 1;
        c->nI = imp[k * 2];
        c->tI = imp[k * 2 + 1];
    }
    w->inv_dt0 = inv_dt0;
    w->new_fixture = new_fixture;
    e->step_count = step_count;
    e->time_passed = time_passed;
    e->done = time_passed > B->p.time_limit;
}

void oracle_set_targets(OBatch* B, int ei, const float* targets /*[T,2]*/)
{
    for (int t = 0; t < B->p.n_targets; ++t) B->e[ei].targets[t] = v2(targets[t * 2], targets[t * 2 + 1]);
}

/* tdm per-agent host state: [E,N,4] = health, cooldown_atk, cooldown_mov_penalty, alive */
void oracle_get_tdm(const OBatch* B, double* st)
{
    int N = B->p.n_agents;
    for (int ei = 0; ei < B->n_envs; ++ei)
        for (int i = 0; i < N; ++i) {
            double* o = st + ((size_t)ei * N + i) * 4;
            const OEnv* e = &B->e[ei];
            o[0] = e->health[i]; o[1] = e->cd_atk[i]; o[2] = e->cd_mov[i]; o[3] = e->alive[i];
        }
}

void oracle_get_env_info(const OBatch* B, int ei, double* out /*[7]*/)
{
    const OEnv* e = &B->e[ei];
    out[0] = e->time_passed; out[1] = e->done; out[2] = e->step_count; out[3] = e->w.inv_dt0;
    out[4] = e->w.last_touching; out[5] = e->w.contact_count; out[6] = e->w.last_peak_contacts;
}

/* ---- thin body-level API: lets tests drive ONE world the way pybox2d is driven, so that the
 * reference's own Python host code can run over it (tests/golden/box2d_shim.py) ------------ */
OBatch* oracle_world_create(double radius, double density, double friction, double linear_damping,
                            int damping_model)
{
    OParams p;
    memset(&p, 0, sizeof(p));
    p.n_agents = O_MAX_BODIES; p.n_targets = 1; p.hz = 60.0; p.radius = radius;   /* room for every body add_body may create */ p.density = density; p.friction = friction;
    p.linear_damping = linear_damping; p.damping_model = damping_model; p.warm_starting = 1;
    return oracle_create(&p, 1);
}
int oracle_world_add_body(OBatch* B, double x, double y, double angle)
{
    if (B->e[0].w.n >= O_MAX_BODIES) return -1;
    B->p.n_agents = B->e[0].w.n + 1;
    return ow_add_body(&B->e[0].w, (float)x, (float)y, (float)angle);
}
void oracle_world_set_angle(OBatch* B, int i, double angle) { ow_set_angle(&B->e[0].w, i, (float)angle); }
double oracle_world_get_angle(const OBatch* B, int i) { return (double)B->e[0].w.b[i].a; }
void oracle_world_apply_force(OBatch* B, int i, double fx, double fy) { ow_apply_force(&B->e[0].w, i, (float)fx, (float)fy); }
void oracle_world_set_active(OBatch* B, int i, int flag) { if (!flag) ow_deactivate(&B->e[0].w, i); }
void oracle_world_set_warm_starting(OBatch* B, int flag) { B->e[0].w.warm_starting = flag; }
void oracle_world_step(OBatch* B, double dt, int vel_iters, int pos_iters) { ow_step(&B->e[0].w, (float)dt, vel_iters, pos_iters); }
int oracle_world_raycast(const OBatch* B, double x1, double y1, double x2, double y2, double* fraction)
{
    float fr = 1.0f;
    int hit = ow_raycast_closest(&B->e[0].w, v2((float)x1, (float)y1), v2((float)x2, (float)y2), &fr);
    if (fraction) *fraction = fr;
    return hit;
}
