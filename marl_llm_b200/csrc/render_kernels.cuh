// render_kernels.cuh — sm_100a rasteriser of swarm_render (include/swarm_b200.h): rgb_array frames of an env's target cells,
// agent trails and agents, straight from the simulator's device buffers.
//
// Pixel rules (DESIGN.md §10, the header's swarm_render): every fp64 operation individually rounded (__d*_rn, never
// contracted), coverage binary, the topmost layer decides a pixel's colour, among agents the largest index wins.  The frames
// are bit-identical to marl_llm_b200/render.py:render_reference.
//
// One CTA per (frame, 32 x 32 pixel tile), 256 threads: lane = pixel column, each thread owns RENDER_ROWS = 4 rows of its
// column (one pixel-centre x, four y).  The frame's primitives (cells, then trail segments, then agents: painter's order) are
// culled against the tile in batches of 256, one per thread, with a bounding-box test widened by one pixel; the survivors are
// compacted into shared memory in ascending order (ballot + per-warp prefix counts); each warp skips the survivors whose box
// misses its 4-row strip (same margin), and every pixel runs the exact test of the others, keeping the colour of the last one
// that covers it.  Each pixel is written once, by its own thread: a warp
// stores 96 contiguous bytes of a row.  No atomics, so the result does not depend on scheduling.
#pragma once
#include <cuda_runtime.h>

#include <stdint.h>

namespace swarm {

constexpr int RENDER_TILE = 32;                                   // tile side in pixels
constexpr int RENDER_THREADS = 256;
constexpr int RENDER_ROWS = RENDER_TILE / (RENDER_THREADS / 32);  // pixel rows per thread
constexpr int RENDER_IDS_PER_LAUNCH = 2048;                       // env ids carried in the kernel parameters (8 KB)
enum { RC_ARENA = 0, RC_OUTSIDE, RC_CELL, RC_TRAIL, RC_AGENT_IN, RC_AGENT_OUT, RC_COUNT };   // palette order of the header

struct RenderParams {
    int W, H, flags, n_a, n_g_pad, count, f0;   // count: frames of the whole call (the trail ring's stride); f0: first frame here
    int cells_ok;                               // the handle has cells and in-shape flags (0 for a flocking handle)
    int trail_cap, trail_len, trail_head;
    double x0, y1, sx, sy;                      // view corner (xmin, ymax) and pixel pitch
    double mx, my;                              // cull margins (one pixel plus rounding slack)
    double ax0, ay1, ax1, ay0;                  // arena: x_min, y_max, x_max, y_min
    double rr_agent, r_agent, w, ww;            // agent disc size_a^2 and its radius; trail half-width and its square
    double half_w, half_h;                      // a trail step longer than this is a periodic wrap
    const double *p;                            // [E][2][n_a]
    const int *in_flags;                        // [E][n_a]
    const double2 *grid;                        // [E][n_g_pad]
    const int *n_g;                             // [E]
    const double *in_thresh;                    // [E]
    const double *trail;                        // [trail_cap][count][2][n_a]
    uint8_t *frames;                            // [count][H][W][3]
    uint8_t palette[RC_COUNT][3];
    int env[RENDER_IDS_PER_LAUNCH];             // env of frame f0 + blockIdx.z
};

__global__ void __launch_bounds__(RENDER_THREADS) k_render(const __grid_constant__ RenderParams P) {
    constexpr int NW = RENDER_THREADS / 32;
    __shared__ double s_a[RENDER_THREADS], s_b[RENDER_THREADS], s_c[RENDER_THREADS], s_d[RENDER_THREADS], s_e[RENDER_THREADS];
    __shared__ double s_ylo[RENDER_THREADS], s_yhi[RENDER_THREADS];     // y extent of the survivor's box
    __shared__ int s_col[RENDER_THREADS];
    __shared__ int s_warp_n[NW];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int f = P.f0 + (int)blockIdx.z, e = P.env[blockIdx.z];
    const int c = (int)blockIdx.x * RENDER_TILE + lane;
    const int r0 = (int)blockIdx.y * RENDER_TILE + warp * RENDER_ROWS;

    // pixel centres: X = x0 + (c + 0.5) sx,  Y = y1 - (r + 0.5) sy; background by the closed arena box
    const double X = __dadd_rn(P.x0, __dmul_rn((double)c + 0.5, P.sx));
    const bool x_in = P.ax0 <= X && X <= P.ax1;
    double Y[RENDER_ROWS];
    int col[RENDER_ROWS];
#pragma unroll
    for (int j = 0; j < RENDER_ROWS; ++j) {
        Y[j] = __dsub_rn(P.y1, __dmul_rn((double)(r0 + j) + 0.5, P.sy));
        col[j] = (x_in && P.ay0 <= Y[j] && Y[j] <= P.ay1) ? RC_ARENA : RC_OUTSIDE;
    }
    // the warp's strip of RENDER_ROWS rows, widened by the cull margin: survivors whose box misses it are skipped by the warp
    const double strip_hi = Y[0] + P.my, strip_lo = Y[RENDER_ROWS - 1] - P.my;

    // the tile's world box, widened by the cull margin (only the exact tests below decide coverage)
    const double tx0 = P.x0 + (double)(blockIdx.x * RENDER_TILE) * P.sx - P.mx;
    const double tx1 = P.x0 + (double)((blockIdx.x + 1) * RENDER_TILE) * P.sx + P.mx;
    const double ty1 = P.y1 - (double)(blockIdx.y * RENDER_TILE) * P.sy + P.my;
    const double ty0 = P.y1 - (double)((blockIdx.y + 1) * RENDER_TILE) * P.sy - P.my;

    const int n_cells = ((P.flags & 1) && P.cells_ok) ? min(P.n_g[e], P.n_g_pad) : 0;
    const int n_seg = ((P.flags & 4) && P.trail_len > 1) ? (P.trail_len - 1) * P.n_a : 0;
    const int n_agents = (P.flags & 2) ? P.n_a : 0;
    const int total = n_cells + n_seg + n_agents;
    const double rr_cell = n_cells ? __dmul_rn(P.in_thresh[e], 0.5) : 0.0;
    const double r_cell = sqrt(rr_cell);
    const double *pe = P.p + (size_t)e * 2 * P.n_a;
    const int first = (P.trail_head - P.trail_len + 1 + P.trail_cap) % max(P.trail_cap, 1);   // ring slot of the oldest sample

    for (int base = 0; base < total; base += RENDER_THREADS) {
        // ---- cull: one primitive per thread; record (a, b, c, d, e, colour) of the ones whose box meets the tile
        const int k = base + tid;
        bool keep = false;
        double a = 0, b = 0, cc = 0, d = 0, ee = 0, ylo = 0, yhi = 0;
        int colour = 0;
        if (k < n_cells) {
            const double2 g = P.grid[(size_t)e * P.n_g_pad + k];
            a = g.x; b = g.y; cc = rr_cell; colour = RC_CELL;
            ylo = b - r_cell; yhi = b + r_cell;
            keep = a + r_cell >= tx0 && a - r_cell <= tx1 && yhi >= ty0 && ylo <= ty1;
        } else if (k < n_cells + n_seg) {
            const int t = k - n_cells, s = t / P.n_a, i = t - s * P.n_a;
            const size_t sa = ((size_t)((first + s) % P.trail_cap) * P.count + f) * 2 * P.n_a + i;
            const size_t sb = ((size_t)((first + s + 1) % P.trail_cap) * P.count + f) * 2 * P.n_a + i;
            const double Ax = P.trail[sa], Ay = P.trail[sa + P.n_a], Bx = P.trail[sb], By = P.trail[sb + P.n_a];
            const double ux = __dsub_rn(Bx, Ax), uy = __dsub_rn(By, Ay);
            a = Ax; b = Ay; cc = ux; d = uy; ee = __dadd_rn(__dmul_rn(ux, ux), __dmul_rn(uy, uy)); colour = RC_TRAIL;
            ylo = fmin(Ay, By) - P.w; yhi = fmax(Ay, By) + P.w;
            keep = fabs(ux) <= P.half_w && fabs(uy) <= P.half_h &&
                   fmax(Ax, Bx) + P.w >= tx0 && fmin(Ax, Bx) - P.w <= tx1 && yhi >= ty0 && ylo <= ty1;
        } else if (k < total) {
            const int i = k - n_cells - n_seg;
            a = pe[i]; b = pe[P.n_a + i]; cc = P.rr_agent;
            colour = (P.cells_ok && (P.in_flags[(size_t)e * P.n_a + i] & 1)) ? RC_AGENT_IN : RC_AGENT_OUT;
            ylo = b - P.r_agent; yhi = b + P.r_agent;
            keep = a + P.r_agent >= tx0 && a - P.r_agent <= tx1 && yhi >= ty0 && ylo <= ty1;
        }
        // ---- compact the survivors in ascending primitive order
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp_n[warp] = __popc(m);
        __syncthreads();
        int off = 0, n = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            const int v = s_warp_n[w];
            off += w < warp ? v : 0;
            n += v;
        }
        if (keep) {
            const int slot = off + __popc(m & ((1u << lane) - 1u));
            s_a[slot] = a; s_b[slot] = b; s_c[slot] = cc; s_d[slot] = d; s_e[slot] = ee; s_col[slot] = colour;
            s_ylo[slot] = ylo; s_yhi[slot] = yhi;
        }
        __syncthreads();
        // ---- exact tests, painter's order
        for (int q = 0; q < n; ++q) {
            if (s_yhi[q] < strip_lo || s_ylo[q] > strip_hi) continue;     // uniform across the warp
            const int cq = s_col[q];
            const double qa = s_a[q], qb = s_b[q], qc = s_c[q];
            if (cq == RC_TRAIL) {            // capsule around A -> A + u: the closest point q = A + t u, t clamped to [0, 1]
                const double qd = s_d[q], ll = s_e[q];
                const double px = __dmul_rn(__dsub_rn(X, qa), qc);
#pragma unroll
                for (int j = 0; j < RENDER_ROWS; ++j) {
                    double t = ll > 0.0 ? __ddiv_rn(__dadd_rn(px, __dmul_rn(__dsub_rn(Y[j], qb), qd)), ll) : 0.0;
                    t = fmin(fmax(t, 0.0), 1.0);
                    const double dx = __dsub_rn(X, __dadd_rn(qa, __dmul_rn(t, qc)));
                    const double dy = __dsub_rn(Y[j], __dadd_rn(qb, __dmul_rn(t, qd)));
                    if (__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) <= P.ww) col[j] = RC_TRAIL;
                }
            } else {                         // disc: dx^2 + dy^2 <= rr
                const double dx = __dsub_rn(X, qa), dx2 = __dmul_rn(dx, dx);
#pragma unroll
                for (int j = 0; j < RENDER_ROWS; ++j) {
                    const double dy = __dsub_rn(Y[j], qb);
                    if (__dadd_rn(dx2, __dmul_rn(dy, dy)) <= qc) col[j] = cq;
                }
            }
        }
        __syncthreads();                     // the next batch overwrites the survivor arrays
    }

    if (c >= P.W) return;
#pragma unroll
    for (int j = 0; j < RENDER_ROWS; ++j) {
        if (r0 + j >= P.H) break;
        uint8_t *o = P.frames + (((size_t)f * P.H + (r0 + j)) * P.W + c) * 3;
        o[0] = P.palette[col[j]][0]; o[1] = P.palette[col[j]][1]; o[2] = P.palette[col[j]][2];
    }
}

}  // namespace swarm
