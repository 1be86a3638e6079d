// macm_lidar.cu -- lidar scans (macm_lidar, include/macm.h): every agent's fan of closest-hit ray casts, cast from
// the bound state.
//
// A block takes one env row.  Its threads stage the env's positions, angles and proxy bits once; each warp then takes
// agents warp, warp + 8, ...  Per agent the warp's lanes first cull the bodies, one lane each, into a list of
// survivors in index order: a body far beyond max_range is dropped, a body whose disc holds or nearly holds the origin
// is kept for every ray, and any other body is kept with the one or two ranges of ray indices its angular interval
// [phi - asin(rho / d), phi + asin(rho / d)] covers.  rho is the radius widened by margins that cover the rounding of
// p2 and of the fp32 test near tangency and at fraction 1 (DESIGN.md section 3, Lidar, gives the argument; the cull
// may only ever keep too much).  Then the rays go 32 at a time, one lane each: the survivors scatter themselves into
// per-ray bit sets with shared-memory atomics (the transpose from bodies to rays), and each lane runs the exact
// b2CircleShape::RayCast of ow_raycast_closest on its set's members in index order -- the oracle's loop with the
// proven misses left out, so the result is the oracle's bit for bit.  A lane's ray is one element of a contiguous
// row: every chunk of 32 rays stores whole lines.
//
// The exact test is fp32 in Box2D's operation order; the library is built with -fmad=false, so nothing is contracted.
// The direction is float64 sin / cos, which can differ from libm's in the last bit: a ray can only differ from the
// oracle where that bit changes the fp32 dx or dy.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <float.h>

#include "macm_sim.h"

namespace {

constexpr int kWarps = 8, kThreads = 32 * kWarps;
constexpr int kMax = MACM_MAX_AGENTS;
constexpr float kPi = 3.14159265f, k2Pi = 6.28318531f;

struct Env {
    float2 pos[kMax];
    float ang[kMax];
    uint32_t proxy[kMax / 32];   // bit j: agent j has a proxy (every Flock agent; a live TDM agent)
};

struct Survivors {
    float sx[kMax], sy[kMax], bb[kMax];   // s = p1 - c and |s|^2 - r^2, as the exact test computes them
    int16_t lo[2][kMax], hi[2][kMax];     // the rays it may hit: [lo0, hi0] and [lo1, hi1], each possibly empty
    uint8_t id[kMax];                     // agent index
    uint32_t cand[32][5];                 // per ray of the chunk: bit q = survivor q is tested (4 words, padded)
};

// bits of the rays r0..r0+31 that lie in [lo, hi]
__device__ __forceinline__ uint32_t span(int lo, int hi, int r0)
{
    const int a = max(lo - r0, 0), b = min(hi - r0, 31);
    return a > b ? 0u : (2u << b) - (1u << a);
}

// ray indices whose angle from the heading o_r lies in [a0, a1]: x(o) = o K + (R - 1) / 2 is r at o_r, and one index
// of slack on each side covers the fp32 evaluation of x
__device__ __forceinline__ void ray_range(float a0, float a1, float K, float half, int nr, int16_t& lo, int16_t& hi)
{
    const float x0 = fminf(fmaxf(a0 * K + half, -2.0f), nr + 1.0f);
    const float x1 = fminf(fmaxf(a1 * K + half, -2.0f), nr + 1.0f);
    lo = (int16_t)max((int)floorf(x0) - 1, 0);
    hi = (int16_t)min((int)ceilf(x1) + 1, nr - 1);
}

__device__ __forceinline__ void store_fraction(void* f, size_t o, float v, int dtype)
{
    if (dtype == MACM_OBS_F32)
        static_cast<float*>(f)[o] = v;
    else if (dtype == MACM_OBS_F16)
        static_cast<__half*>(f)[o] = __float2half_rn(v);
    else
        static_cast<__nv_bfloat16*>(f)[o] = __float2bfloat16_rn(v);
}

__global__ void __launch_bounds__(kThreads)
macm_lidar_kernel(const RenderConst R, const int32_t* __restrict__ envs, const int nr, const double L, const double fov,
                  void* __restrict__ fraction, int32_t* __restrict__ hit, const int dtype)
{
    __shared__ Env S;
    __shared__ Survivors Wp[kWarps];
    const int b = blockIdx.x, N = R.N;
    const int e = envs ? envs[b] : b;
    const size_t row = (size_t)b * N * nr;
    if (!(e >= 0 && e < R.E)) {   // a bad env index: a row of misses, and nothing is read for it
        for (size_t k = threadIdx.x; k < (size_t)N * nr; k += kThreads) {
            store_fraction(fraction, row + k, 1.0f, dtype);
            if (hit) hit[row + k] = -1;
        }
        return;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    {
        const int k = threadIdx.x;   // kThreads >= MACM_MAX_AGENTS: one agent per thread
        bool proxy = false;
        if (k < N) {
            const size_t a = (size_t)e * N + k;
            const float4 pv = R.posvel[a];
            S.pos[k] = make_float2(pv.x, pv.y);
            S.ang[k] = R.angsleep[a].x;
            proxy = R.kind == MACM_ENV_FLOCK || (__float_as_int(R.tdm[a].w) & 1);
        }
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, proxy);
        if (warp < kMax / 32 && lane == 0) S.proxy[warp] = m;
    }
    __syncthreads();

    Survivors& W = Wp[warp];
    const float r = (float)R.radius, r2 = r * r, Lf = (float)L;
    const float K = (float)fmin((double)nr / fov, 1e30), half = 0.5f * (float)(nr - 1);
    for (int i = warp; i < N; i += kWarps) {
        const float2 p1 = S.pos[i];
        const float ai = S.ang[i];
        // e: how far the rounding of p2 = p1 + (dx, dy) can move the segment within reach of a hit; delta: the error of
        // the fp32 angles below (atan2f, asinf, the heading, the wrap) and of the fp32 direction (dx, dy)
        const float eps = 0x1p-20f * (1.0f + 2.0f * r / Lf) * (fabsf(p1.x) + fabsf(p1.y) + Lf);
        const float delta = 0x1p-16f + 0x1p-18f * fabsf(ai);
        int ns = 0;
        for (int base = 0; base < N; base += 32) {
            const int j = base + lane;
            bool keep = false;
            float sx = 0.0f, sy = 0.0f, bq = 0.0f;
            int16_t lo0 = 0, hi0 = -1, lo1 = 0, hi1 = -1;
            if (j < N && (S.proxy[j >> 5] >> (j & 31) & 1u)) {
                const float2 c = S.pos[j];
                sx = p1.x - c.x;
                sy = p1.y - c.y;
                const float d2 = sx * sx + sy * sy;
                bq = d2 - r2;
                const float d = sqrtf(d2);
                // rho: the radius widened by the p2 rounding and by the cancellation of sigma = c^2 - rr bb, whose
                // error is a few ulp of rr (|s|^2 + r^2)
                const float rm = r * (1.0f + 0x1p-16f) + eps;
                const float rho = sqrtf(rm * rm + 0x1p-18f * (d2 + r2));
                if (!(rho <= FLT_MAX) || d <= rho + eps || K >= 1e30f) {
                    keep = true;   // the disc holds or nearly holds the origin (or no bound is finite): every ray
                    lo0 = 0;
                    hi0 = (int16_t)(nr - 1);
                } else if (d <= Lf * (1.0f + 0x1p-18f) + rho + eps) {
                    const float w = asinf(rho / d) + delta;
                    if (w >= kPi) {
                        keep = true;
                        lo0 = 0;
                        hi0 = (int16_t)(nr - 1);
                    } else {
                        float psi = atan2f(-sy, -sx) - ai;   // the body's direction from the heading
                        psi -= k2Pi * rintf(psi * (1.0f / k2Pi));
                        float a0 = psi - w;
                        if (a0 < -kPi) a0 += k2Pi;
                        else if (a0 >= kPi) a0 -= k2Pi;
                        const float a1 = a0 + 2.0f * w;      // [a0, a1] from a0 in [-pi, pi): also reaches the rays
                        ray_range(a0, a1, K, half, nr, lo0, hi0);                // near -pi from above +pi
                        ray_range(a0 - k2Pi, a1 - k2Pi, K, half, nr, lo1, hi1);
                        keep = lo0 <= hi0 || lo1 <= hi1;
                    }
                }
            }
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, keep);
            if (keep) {
                const int q = ns + __popc(m & ((1u << lane) - 1u));
                W.sx[q] = sx; W.sy[q] = sy; W.bb[q] = bq; W.id[q] = (uint8_t)j;
                W.lo[0][q] = lo0; W.hi[0][q] = hi0; W.lo[1][q] = lo1; W.hi[1][q] = hi1;
            }
            ns += __popc(m);
        }
        __syncwarp();

        const size_t out = row + (size_t)i * nr;
        for (int r0 = 0; r0 < nr; r0 += 32) {
            const int ray = r0 + lane;
            float rx = 0.0f, ry = 0.0f, rr = 0.0f;
            if (ray < nr) {
                const double o = fov * ((double)(2 * ray + 1 - nr) / (double)(2 * nr));
                double sn, cs;
                sincos((double)ai + o, &sn, &cs);
                const float dx = (float)(L * cs), dy = (float)(L * sn);
                const float p2x = p1.x + dx, p2y = p1.y + dy;
                rx = p2x - p1.x;
                ry = p2y - p1.y;
                rr = rx * rx + ry * ry;
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) W.cand[lane][g] = 0u;
            __syncwarp();
            for (int base = 0; base < ns; base += 32) {
                const int q = base + lane;
                if (q < ns) {
                    uint32_t m = span(W.lo[0][q], W.hi[0][q], r0) | span(W.lo[1][q], W.hi[1][q], r0);
                    for (; m; m &= m - 1u) atomicOr(&W.cand[__ffs(m) - 1][base >> 5], 1u << lane);
                }
            }
            __syncwarp();
            // b2CircleShape::RayCast (ow_raycast_closest): smallest fraction, lowest index among equal ones
            float best = 1.0f;
            int id = -1;
            if (ray < nr && !(rr < B2_EPSILON)) {
                for (int g = 0; 32 * g < ns; ++g) {
                    for (uint32_t m = W.cand[lane][g]; m; m &= m - 1u) {
                        const int q = 32 * g + __ffs(m) - 1;
                        const float sx = W.sx[q], sy = W.sy[q], bq = W.bb[q];
                        const float c = sx * rx + sy * ry;
                        const float sigma = c * c - rr * bq;
                        if (sigma < 0.0f) continue;
                        float a = -(c + sqrtf(sigma));
                        if (0.0f <= a && a <= 1.0f * rr) {
                            a /= rr;
                            if (id < 0 || a < best) { id = W.id[q]; best = a; }
                        }
                    }
                }
            }
            if (ray < nr) {
                store_fraction(fraction, out + ray, best, dtype);
                if (hit) hit[out + ray] = id;
            }
            __syncwarp();   // the bit sets are rebuilt for the next chunk, the survivors for the next agent
        }
    }
}

}  // namespace

cudaError_t macm_launch_lidar(const RenderConst& R, const macm_lidar_args& a, int obs_dtype, cudaStream_t s)
{
    macm_lidar_kernel<<<(unsigned)a.n_envs, kThreads, 0, s>>>(R, a.envs, a.n_rays, a.max_range, a.fov, a.fraction,
                                                              a.hit, obs_dtype);
    return cudaGetLastError();
}
