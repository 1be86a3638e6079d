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

}  // namespace

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
