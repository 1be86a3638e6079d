// macm_render.cu -- top-down RGB frames of envs of the batch (macm_render, include/macm.h), drawn from the bound state.
//
// A block serves one frame, or a chunk of kTilesPerBlock warp tiles of a large one.  Its threads first stage the
// frame's primitives in shared memory, one thread each: agents 0..N-1 then (Flock) targets 0..T-1, which is the
// painter's order.  Each warp then takes tiles of 4 rows x 32 columns, culls the primitive list against the tile with
// ballots (keeping the order), and each lane walks the surviving list from the last primitive to the first for its
// four horizontally adjacent pixels, stopping at the first cover of each.  Four pixels are 12 bytes: three 32-bit
// stores when rows are whole groups of four pixels.
//
// The geometry is float64, evaluated in the same order as the float64 restatement of the drawing rules that the
// tests hold the kernel to (the library is built with -fmad=false, so nothing is contracted): a pixel can only differ
// from it where a predicate sits at its threshold to within the last bits of sin / cos.  B200 issues float64 at half
// the float32 rate; DESIGN.md (section 3, Frames) gives the measured cost and what bounds it.
#include <float.h>
#include <limits.h>

#include "macm_sim.h"

namespace {

constexpr int kWarps = 8, kThreads = 32 * kWarps;
constexpr int kTileRows = 4, kTileCols = 32;           // one warp: 4 rows x 8 lanes of 4 pixels
constexpr int kTilesPerBlock = 64;                     // 8192 pixels: an 84 x 84 frame is one block
constexpr int kMaxPrims = MACM_MAX_AGENTS + MACM_MAX_TARGETS;

struct Prims {
    double cu[kMaxPrims], cv[kMaxPrims];   // centre, pixels
    double r2[kMaxPrims], in2[kMaxPrims];  // rho^2 and the outline's inner bound (rho - 1)^2, or -1 when rho < 1
    double ux[kMaxPrims], uy[kMaxPrims];   // agents: heading (cos angle, -sin angle) in pixel axes
    double len[kMaxPrims];                 // agents: rho, the length of the heading axis
    float4 box[kMaxPrims];                 // u0 v0 u1 v1 holding every pixel centre the primitive can cover
    uint32_t col[kMaxPrims];               // r | g << 8 | b << 16
    uint8_t list[kWarps][kMaxPrims];       // per warp: the primitives that meet its tile, in painter's order
};

__global__ void __launch_bounds__(kThreads)
macm_render_kernel(const RenderConst R, const int H, const int W, const int32_t* __restrict__ envs,
                   const float* __restrict__ views, const uint8_t* __restrict__ palette, uint8_t* __restrict__ out,
                   const int chunks, const int tiles_x, const int tiles)
{
    __shared__ Prims S;
    const int b = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
    const int e = envs ? envs[b] : b;
    const float cx = views[3 * b], cy = views[3 * b + 1], hw = views[3 * b + 2];
    // a bad env index or view leaves the frame black, and nothing is read for it
    const bool ok = e >= 0 && e < R.E && hw > 0.0f && hw <= FLT_MAX;
    const int P = ok ? R.N + R.T : 0;
    const double s = (double)W / (2.0 * (double)hw), w2 = (double)W * 0.5, h2 = (double)H * 0.5;

    for (int k = threadIdx.x; k < P; k += kThreads) {
        double x, y, rho;
        uint32_t col;
        if (k < R.N) {
            const size_t a = (size_t)e * R.N + k;
            const float4 pv = R.posvel[a];
            const int alt = R.kind == MACM_ENV_FLOCK ? R.collided[a] != 0 : !(__float_as_int(R.tdm[a].w) & 1);
            const uint8_t* c = palette + (2 * k + alt) * 3;
            double sn, cs;
            sincos((double)R.angsleep[a].x, &sn, &cs);
            x = pv.x; y = pv.y; rho = R.radius * s;
            col = (uint32_t)c[0] | (uint32_t)c[1] << 8 | (uint32_t)c[2] << 16;
            S.ux[k] = cs; S.uy[k] = -sn; S.len[k] = rho;
        } else {
            const float2 t = R.targets[(size_t)e * R.T + (k - R.N)];
            x = t.x; y = t.y; rho = R.reward_radius * s;
            col = 0xFFFFFFu;
        }
        const double u = (x - (double)cx) * s + w2, v = ((double)cy - y) * s + h2;
        S.cu[k] = u; S.cv[k] = v;
        S.r2[k] = rho * rho;
        S.in2[k] = rho >= 1.0 ? (rho - 1.0) * (rho - 1.0) : -1.0;
        S.col[k] = col;
        const double m = rho + 0.75;   // the heading axis reaches 0.5 px past the rim
        S.box[k] = make_float4(__double2float_rd(u - m), __double2float_rd(v - m), __double2float_ru(u + m),
                               __double2float_ru(v + m));
    }
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* list = S.list[warp];
    const bool words = W % 4 == 0 && ((uintptr_t)out & 3) == 0;
    for (int m = 0; m < kTilesPerBlock / kWarps; ++m) {
        const int tile = chunk * kTilesPerBlock + m * kWarps + warp;
        if (tile >= tiles) break;
        const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
        const float u0 = tx * kTileCols + 0.5f, u1 = u0 + (kTileCols - 1), v0 = ty * kTileRows + 0.5f,
                    v1 = v0 + (kTileRows - 1);
        int n = 0;
        for (int base = 0; base < P; base += 32) {
            const int k = base + lane;
            bool hit = false;
            if (k < P) {
                const float4 bx = S.box[k];
                hit = bx.x <= u1 && bx.z >= u0 && bx.y <= v1 && bx.w >= v0;
            }
            const unsigned mask = __ballot_sync(0xFFFFFFFFu, hit);
            if (hit) list[n + __popc(mask & ((1u << lane) - 1u))] = (uint8_t)k;
            n += __popc(mask);
        }
        __syncwarp();

        const int row = ty * kTileRows + (lane >> 3), col0 = tx * kTileCols + (lane & 7) * 4;
        uint32_t px[4] = {0u, 0u, 0u, 0u};
        unsigned todo = 0u;   // pixels of this lane inside the frame that no primitive has covered yet
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (row < H && col0 + q < W) todo |= 1u << q;
        const double py = row + 0.5;
        for (int j = n - 1; j >= 0 && todo; --j) {
            const int k = list[j];
            const double cu = S.cu[k], dy = py - S.cv[k], r2 = S.r2[k], in2 = S.in2[k];
            const uint32_t c = S.col[k];
            const bool agent = k < R.N;
            const double ux = agent ? S.ux[k] : 0.0, uy = agent ? S.uy[k] : 0.0, len = agent ? S.len[k] : 0.0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (!(todo >> q & 1u)) continue;
                const double dx = (col0 + q + 0.5) - cu;
                const double d2 = dx * dx + dy * dy;
                bool hit = false;
                uint32_t hc = c;
                if (agent) {
                    double t = dx * ux + dy * uy;
                    t = t < 0.0 ? 0.0 : (t > len ? len : t);
                    const double ex = dx - t * ux, ey = dy - t * uy;
                    if (ex * ex + ey * ey <= 0.25) {
                        hit = true;                       // heading axis
                    } else if (d2 <= r2) {
                        hit = true;                       // outline, or the fill at half the colour
                        if (!(d2 > in2)) hc = (c >> 1) & 0x7F7F7Fu;
                    }
                } else {
                    hit = d2 <= r2 && d2 > in2;           // target ring
                }
                if (hit) { px[q] = hc; todo &= ~(1u << q); }
            }
        }
        __syncwarp();   // the list is rebuilt for the next tile

        if (row < H && col0 < W) {
            const size_t o = ((size_t)b * H + row) * W + col0;
            if (words) {   // W % 4 == 0: the four pixels are in the row and start on a 4-byte boundary
                uint32_t* w = reinterpret_cast<uint32_t*>(out + o * 3);
                w[0] = px[0] | px[1] << 24;
                w[1] = px[1] >> 8 | px[2] << 16;
                w[2] = px[2] >> 16 | px[3] << 8;
            } else {
                for (int q = 0; q < 4 && col0 + q < W; ++q) {
                    uint8_t* p = out + (o + q) * 3;
                    p[0] = (uint8_t)px[q]; p[1] = (uint8_t)(px[q] >> 8); p[2] = (uint8_t)(px[q] >> 16);
                }
            }
        }
    }
}

// ---- agent-centred frames (macm_render_agents) ------------------------------------------------------------------
//
// A block takes one env row and a chunk of its jobs: a job is one agent's frame, or a group of kJobTiles warp tiles
// of a large one.  The block's threads stage the env once -- positions, float64 cos / sin of every agent's angle (once
// per agent, not once per agent per frame) and the colour each primitive shows -- and each warp then takes jobs
// w, w + 8, ... of the chunk.  Per job the warp's lanes transform the primitives into the frame, one lane each, and
// cull them against the frame with ballots that keep the painter's order; for a frame of more than one tile, each
// tile culls that list again.  Tiles are 32 lanes of 4 horizontally adjacent pixels, as wide as the frame needs up to
// 32 pixels (16 x 16: 2 tiles of 8 rows x 16 columns), so small frames keep every lane busy.  Each lane walks the list
// from the last primitive to the first, evaluating the predicates of macm_render_kernel only for the primitives whose
// bounding box holds one of its four pixel centres.  A tile whose rows are one run in memory is stored contiguously.

constexpr int kJobsPerBlock = 64;   // one block per env row up to 64 agents
constexpr int kJobTiles = 64;       // a job covers up to 8192 pixels

struct AgentEnv {
    float2 pos[kMaxPrims];              // world centres, agents then targets
    double cs[MACM_MAX_AGENTS], sn[MACM_MAX_AGENTS];
    uint32_t col[kMaxPrims];
};

struct AgentWarp {
    double cu[kMaxPrims], cv[kMaxPrims];   // pixel centres in this warp's frame of the primitives that meet it
    float4 box[kMaxPrims];
    uint8_t prim[kMaxPrims];                // the primitive behind each entry, in painter's order
    uint8_t list[kMaxPrims];                // entries that meet the current tile
};

__global__ void __launch_bounds__(kThreads, 3)   // 80 registers, no spills: three blocks per SM
macm_render_agents_kernel(const RenderConst R, const int H, const int W, const double s,
                          const int32_t* __restrict__ envs, const uint8_t* __restrict__ palette,
                          uint8_t* __restrict__ out, const int chunks, const int jobs_per_frame, const int gx,
                          const int tiles_x, const int tiles)
{
    __shared__ AgentEnv S;
    __shared__ AgentWarp Wp[kWarps];
    const int b = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
    const int e = envs ? envs[b] : b;
    // a bad env index gives N black frames, and nothing is read for them
    const bool ok = e >= 0 && e < R.E;
    const int P = ok ? R.N + R.T : 0;
    const double w2 = (double)W * 0.5, h2 = (double)H * 0.5;
    const double rhoA = R.radius * s, rhoT = R.reward_radius * s;

    for (int k = threadIdx.x; k < P; k += kThreads) {
        if (k < R.N) {
            const size_t a = (size_t)e * R.N + k;
            const float4 pv = R.posvel[a];
            const int alt = R.kind == MACM_ENV_FLOCK ? R.collided[a] != 0 : !(__float_as_int(R.tdm[a].w) & 1);
            const uint8_t* c = palette + (2 * k + alt) * 3;
            sincos((double)R.angsleep[a].x, &S.sn[k], &S.cs[k]);
            S.pos[k] = make_float2(pv.x, pv.y);
            S.col[k] = (uint32_t)c[0] | (uint32_t)c[1] << 8 | (uint32_t)c[2] << 16;
        } else {
            S.pos[k] = R.targets[(size_t)e * R.T + (k - R.N)];
            S.col[k] = 0xFFFFFFu;
        }
    }
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    AgentWarp& A = Wp[warp];
    const int rows = 32 / gx, cols = 4 * gx;    // one tile
    const bool words = W % 4 == 0 && ((uintptr_t)out & 3) == 0;
    const double r2A = rhoA * rhoA, in2A = rhoA >= 1.0 ? (rhoA - 1.0) * (rhoA - 1.0) : -1.0;
    const double r2T = rhoT * rhoT, in2T = rhoT >= 1.0 ? (rhoT - 1.0) * (rhoT - 1.0) : -1.0;
    const int jobs = R.N * jobs_per_frame;
    for (int job = chunk * kJobsPerBlock + warp; job < jobs && job < (chunk + 1) * kJobsPerBlock; job += kWarps) {
        const int i = job / jobs_per_frame, group = job - i * jobs_per_frame;
        double ci = 0.0, si = 0.0;
        int n = 0;   // entries of the frame list
        if (ok) {
            const float2 c = S.pos[i];
            const double cx = c.x, cy = c.y;
            ci = S.cs[i]; si = S.sn[i];
            for (int base = 0; base < P; base += 32) {
                const int k = base + lane;
                bool hit = false;
                double u = 0.0, v = 0.0;
                float4 bx;
                if (k < P) {
                    const double dx = (double)S.pos[k].x - cx, dy = (double)S.pos[k].y - cy;
                    u = w2 + s * (dx * si - dy * ci);
                    v = h2 - s * (dx * ci + dy * si);
                    const double m = (k < R.N ? rhoA : rhoT) + 0.75;   // the heading axis reaches 0.5 px past the rim
                    bx = make_float4(__double2float_rd(u - m), __double2float_rd(v - m), __double2float_ru(u + m),
                                     __double2float_ru(v + m));
                    hit = bx.x <= W - 0.5f && bx.z >= 0.5f && bx.y <= H - 0.5f && bx.w >= 0.5f;
                }
                const unsigned mask = __ballot_sync(0xFFFFFFFFu, hit);
                if (hit) {
                    const int q = n + __popc(mask & ((1u << lane) - 1u));
                    A.cu[q] = u; A.cv[q] = v; A.box[q] = bx; A.prim[q] = (uint8_t)k;
                }
                n += __popc(mask);
            }
            __syncwarp();
        }

        const int t_end = min(tiles, (group + 1) * kJobTiles);
        for (int tile = group * kJobTiles; tile < t_end; ++tile) {
            const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
            const int row = ty * rows + lane / gx, col0 = tx * cols + (lane % gx) * 4;
            int m = n;
            const uint8_t* list = nullptr;   // nullptr: the frame list itself
            if (tiles > 1) {
                const float u0 = tx * cols + 0.5f, u1 = u0 + (cols - 1), v0 = ty * rows + 0.5f, v1 = v0 + (rows - 1);
                m = 0;
                for (int base = 0; base < n; base += 32) {
                    const int q = base + lane;
                    bool hit = false;
                    if (q < n) {
                        const float4 bx = A.box[q];
                        hit = bx.x <= u1 && bx.z >= u0 && bx.y <= v1 && bx.w >= v0;
                    }
                    const unsigned mask = __ballot_sync(0xFFFFFFFFu, hit);
                    if (hit) A.list[m + __popc(mask & ((1u << lane) - 1u))] = (uint8_t)q;
                    m += __popc(mask);
                }
                __syncwarp();
                list = A.list;
            }

            uint32_t px[4] = {0u, 0u, 0u, 0u};
            unsigned todo = 0u;
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (row < H && col0 + q < W) todo |= 1u << q;
            const double py = row + 0.5;
            const float pu0 = col0 + 0.5f, pu1 = col0 + 3.5f, pv = row + 0.5f;
            // the list in chunks of 32 from its end: each lane first marks the entries whose box holds one of its
            // pixel centres, then evaluates only those, the last first -- lanes run their own entries side by side
            for (int base = (m - 1) & ~31; base >= 0 && todo; base -= 32) {
                unsigned hits = 0u;
                const int cnt = min(32, m - base);
                for (int t = 0; t < cnt; ++t) {
                    const float4 bx = A.box[list ? list[base + t] : base + t];
                    if (bx.x <= pu1 && bx.z >= pu0 && bx.y <= pv && bx.w >= pv) hits |= 1u << t;
                }
                while (hits && todo) {
                    const int t = 31 - __clz(hits);
                    hits &= ~(1u << t);
                    const int q = list ? list[base + t] : base + t;
                    const int k = A.prim[q];
                    const double cu = A.cu[q], dy = py - A.cv[q];
                    const bool agent = k < R.N;
                    const double r2 = agent ? r2A : r2T, in2 = agent ? in2A : in2T;
                    const uint32_t c = S.col[k];
                    double ux = 0.0, uy = 0.0;
                    if (agent) {
                        const double ck = S.cs[k], sk = S.sn[k];
                        ux = ck * si - sk * ci;
                        uy = -(ck * ci + sk * si);
                    }
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        if (!(todo >> p & 1u)) continue;
                        const double dx = (col0 + p + 0.5) - cu;
                        const double d2 = dx * dx + dy * dy;
                        bool hit = false;
                        uint32_t hc = c;
                        if (agent) {
                            double tt = dx * ux + dy * uy;
                            tt = tt < 0.0 ? 0.0 : (tt > rhoA ? rhoA : tt);
                            const double ex = dx - tt * ux, ey = dy - tt * uy;
                            if (ex * ex + ey * ey <= 0.25) {
                                hit = true;                       // heading axis
                            } else if (d2 <= r2) {
                                hit = true;                       // outline, or the fill at half the colour
                                if (!(d2 > in2)) hc = (c >> 1) & 0x7F7F7Fu;
                            }
                        } else {
                            hit = d2 <= r2 && d2 > in2;           // target ring
                        }
                        if (hit) { px[p] = hc; todo &= ~(1u << p); }
                    }
                }
            }
            __syncwarp();   // the tile list is rebuilt for the next tile

            const size_t frame = ((size_t)b * R.N + i) * H;
            if (words && cols == W) {
                // the tile's rows are one run of 96 words in memory: shuffle them so that each store is contiguous
                const uint32_t w0 = px[0] | px[1] << 24, w1 = px[1] >> 8 | px[2] << 16, w2 = px[2] >> 16 | px[3] << 8;
                uint32_t* run = reinterpret_cast<uint32_t*>(out + (frame + ty * rows) * W * 3);
                const int nwords = min(rows, H - ty * rows) * W * 3 / 4;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const int w = 32 * r + lane, src = w / 3, part = w - 3 * src;
                    const uint32_t a0 = __shfl_sync(0xFFFFFFFFu, w0, src), a1 = __shfl_sync(0xFFFFFFFFu, w1, src),
                                   a2 = __shfl_sync(0xFFFFFFFFu, w2, src);
                    if (w < nwords) run[w] = part == 0 ? a0 : (part == 1 ? a1 : a2);
                }
            } else if (row < H && col0 < W) {
                const size_t o = (frame + row) * W + col0;
                if (words) {   // W % 4 == 0: the four pixels are in the row and start on a 4-byte boundary
                    uint32_t* w = reinterpret_cast<uint32_t*>(out + o * 3);
                    w[0] = px[0] | px[1] << 24;
                    w[1] = px[1] >> 8 | px[2] << 16;
                    w[2] = px[2] >> 16 | px[3] << 8;
                } else {
                    for (int p = 0; p < 4 && col0 + p < W; ++p) {
                        uint8_t* d = out + (o + p) * 3;
                        d[0] = (uint8_t)px[p]; d[1] = (uint8_t)(px[p] >> 8); d[2] = (uint8_t)(px[p] >> 16);
                    }
                }
            }
        }
        __syncwarp();   // the frame list is rebuilt for the next job
    }
}

}  // namespace

cudaError_t macm_launch_render_agents(const RenderConst& R, const macm_agent_frames_args& a, cudaStream_t s)
{
    // tile: 32 lanes of 4 pixels, gx lanes across (the least power of two that spans the row, at most 8) and 32 / gx down
    int gx = 1;
    while (gx < 8 && 4 * gx < a.width) gx *= 2;
    const int tiles_x = (a.width + 4 * gx - 1) / (4 * gx), tiles_y = (a.height + 32 / gx - 1) / (32 / gx);
    const int tiles = tiles_x * tiles_y, jobs_per_frame = (tiles + kJobTiles - 1) / kJobTiles;
    const int chunks = (R.N * jobs_per_frame + kJobsPerBlock - 1) / kJobsPerBlock;
    const long long blocks = (long long)a.n_envs * chunks;
    if (blocks > INT_MAX) return cudaErrorInvalidValue;
    const double scale = (double)a.width / (2.0 * a.half_width);
    macm_render_agents_kernel<<<(unsigned)blocks, kThreads, 0, s>>>(R, a.height, a.width, scale, a.envs, a.palette,
                                                                    a.out, chunks, jobs_per_frame, gx, tiles_x, tiles);
    return cudaGetLastError();
}

cudaError_t macm_launch_render(const RenderConst& R, const macm_render_args& a, cudaStream_t s)
{
    const int tiles_x = (a.width + kTileCols - 1) / kTileCols, tiles_y = (a.height + kTileRows - 1) / kTileRows;
    const int tiles = tiles_x * tiles_y, chunks = (tiles + kTilesPerBlock - 1) / kTilesPerBlock;
    const long long blocks = (long long)a.n_frames * chunks;
    if (blocks > INT_MAX) return cudaErrorInvalidValue;
    macm_render_kernel<<<(unsigned)blocks, kThreads, 0, s>>>(R, a.height, a.width, a.envs, a.views, a.palette, a.out,
                                                             chunks, tiles_x, tiles);
    return cudaGetLastError();
}
