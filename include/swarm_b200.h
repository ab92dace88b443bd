/*
 * swarm_b200.h — C ABI of the B200-native batched simulator for the MARL-LLM assembly env step path.
 *
 * One shared library (marl_llm_b200/lib/libswarm_b200.so, also reachable as libAssemblyEnv.so)
 * exports these groups of entry points (the first two below; (3)-(6) further down), all `extern "C"`, plain pointers and sizes only:
 *
 *  (1) LEGACY, stateless, HOST pointers — the five symbols the reference Python env binds with ctypes
 *      (cus_gym/gym/envs/customized_envs/envs_cplus/c_lib.py:11-22 loads build/libAssemblyEnv.so;
 *      assembly.py:234-255, 357-380, 460-466, 495-504, 613-624 call them).  Same names, argument order,
 *      layouts, in-place output convention and `void` return as AssemblyEnv.h:13-58,64-81,98-109, so the
 *      reference's assembly.py runs unchanged on top of this library.  Each call copies its inputs to the
 *      GPU, runs the corresponding sm_100a kernel for a batch of one env, and copies the outputs back.
 *
 *  (2) BATCHED, handle based, DEVICE-resident — the product path: E independent envs stepped by ONE fused
 *      kernel launch per step (forces + walls + integrator + k-NN + grid scan + occupancy + observation
 *      packing + reward + next prior).  Not in the reference (it has no vector env, SURVEY.md §0.1); per-env
 *      layouts are identical to the reference's so that obs[e] == the reference's obs for that env.
 *
 * Reference abbreviations used below:
 *   HDR = cus_gym/gym/envs/customized_envs/envs_cplus/src/AssemblyEnv.h
 *   CPP = cus_gym/gym/envs/customized_envs/envs_cplus/src/AssemblyEnv.cpp
 *   ENV = cus_gym/gym/envs/customized_envs/assembly.py
 */
#ifndef SWARM_B200_H
#define SWARM_B200_H

#include <stdint.h>
#include <stdbool.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ============================================================================================
 * (1) Legacy entry points (HOST pointers, stateless).  A CUDA failure inside one of these cannot be
 *     reported through the reference's void signatures: it is printed to stderr and the process aborts
 *     (there is deliberately NO CPU fallback).
 * ============================================================================================ */

/* replaces HDR:13-34 / CPP:18-351; bound at ENV:234-255.
 * p, dp, heading: [dim][n_a] f64; obs: [obs_dim_agent][n_a] f64 (out); boundary_pos: [4] = xmin,ymax,xmax,ymin;
 * grid_center: [dim][n_g] f64; neighbor_index: [n_a][topo_nei_max] i32 (out); in_flags: [n_a] i32 (out);
 * sensed_index: [n_a][num_obs_grid_max] i32 (out); occupied_index: [n_a][num_occupied_grid_max] i32 (out);
 * condition: bool[4] = is_periodic, is_Cartesian, is_con_self_state, is_feature_norm (the last is never read
 * by the reference either, CPP:80,88,103,294).  All outputs are fully written (the caller's -1 / 0 pre-fill
 * of ENV:227-231 is not relied upon). */
void _get_observation(double *p, double *dp, double *heading, double *obs, double *boundary_pos,
                      double *grid_center, int *neighbor_index, int *in_flags, int *sensed_index,
                      int *occupied_index, double d_sen, double r_avoid, double l_cell, double Vel_max,
                      int topo_nei_max, int num_obs_grid_max, int num_occupied_grid_max, int n_a, int n_g,
                      int obs_dim_agent, int dim, bool *condition);

/* replaces HDR:35-58 / CPP:354-626; bound at ENV:357-380.  reward: [1][n_a] f64 (out).
 * condition: bool[5] = is_periodic, is_Cartesian, penalize_entering, penalize_interaction, penalize_exploration.
 * act, heading, occupied_index, is_collide_b2b, is_collide_b2w, coefficients are accepted and ignored exactly as
 * the live branch of the reference ignores them (CPP:452-559). */
void _get_reward(double *p, double *dp, double *heading, double *act, double *reward, double *boundary_pos,
                 double *grid_center, int *neighbor_index, int *in_flags, int *sensed_index, int *occupied_index,
                 double d_sen, double r_avoid, double l_cell, int topo_nei_max, int num_obs_grid_max,
                 int num_occupied_grid_max, int n_a, int n_g, int dim, bool *condition, bool *is_collide_b2b,
                 bool *is_collide_b2w, double *coefficients);

/* replaces HDR:64-73 / CPP:735-815; bound at ENV:495-504.  sf_b2b: [dim][n_a] f64 (out);
 * d_b2b_edge, d_b2b_center: [n_a][n_a] f64 and is_collide_b2b: [n_a][n_a] bool, as produced by ENV:442-457. */
void _sf_b2b_all(double *p, double *sf_b2b, double *d_b2b_edge, bool *is_collide_b2b, double *boundary_pos,
                 double *d_b2b_center, int n_a, int dim, double k_ball, bool is_periodic);

/* replaces HDR:75-81 / CPP:817-855; bound at ENV:460-466.  r: [n_a]; d_b2w: [4][n_a] f64 (out);
 * isCollision: [4][n_a] bool (out). */
void _get_dist_b2w(double *p, double *r, double *d_b2w, bool *isCollision, int dim, int n_a, double *boundary_pos);

/* replaces HDR:98-109 / CPP:1061-1196; bound at ENV:613-624.  a_prior: [dim][n_a] f64 (out). */
void calculateActionPrior(double *p, double *dp, double *a_prior, double *grid_center, int *neighbor_index,
                          double d_sen, double r_avoid, double l_cell, int topo_nei_max, int n_a, int n_g, int dim);

/* ============================================================================================
 * (2) Batched, device-resident simulator.
 * ============================================================================================ */

typedef struct swarm_sim swarm_sim;   /* opaque */

enum {
    SWARM_OK = 0,
    SWARM_ERR_INVALID = 1,       /* bad argument / inconsistent sizes                      */
    SWARM_ERR_UNSUPPORTED = 2,   /* valid in the reference but outside this build's limits  */
    SWARM_ERR_CUDA = 3,          /* a CUDA call failed; see swarm_last_error()              */
    SWARM_ERR_NO_DEVICE = 4      /* no usable sm_100 device: there is no CPU fallback       */
};

enum { SWARM_F64 = 0, SWARM_F32 = 1 };
enum { SWARM_OBS_REFERENCE = 0, SWARM_OBS_AGENT_MAJOR = 1 };
enum { SWARM_VARIANT_ASSEMBLY = 0, SWARM_VARIANT_FLOCKING = 1 };

/* Everything ENV:27-81,93-138,193-199 fixes per env class; per-env quantities (n_g, l_cell, grid) are set
 * with swarm_set_grid(). */
typedef struct swarm_config {
    int32_t struct_size;            /* sizeof(swarm_config), ABI check                                 */
    int32_t device;                 /* CUDA device ordinal                                             */
    int32_t num_envs;               /* E                                                               */
    int32_t n_a;                    /* agents per env (<= 1024)                       ENV:93           */
    int32_t n_g_max;                /* capacity in cells per env (any n_g <= n_g_max)  ENV:179          */
    int32_t topo_nei_max;           /* must be 6                                       ENV:34           */
    int32_t num_obs_grid_max;       /* 80                                              ENV:128          */
    int32_t num_occupied_grid_max;  /* 200                                             ENV:130          */
    int32_t is_con_self_state;      /* obs_dim 192 (1) or 188 (0)                      ENV:107,801      */
    int32_t is_periodic;            /* !is_boundary: periodic wrap instead of walls     ENV:99-103,651   */
    int32_t want_prior;             /* training_method == 'llm_rl'                     ENV:605          */
    int32_t out_dtype;              /* SWARM_F64 (reference dtype) or SWARM_F32 for obs/reward/a_prior  */
    int32_t emit_indices;           /* also write sensed_index / occupied_index every step             */
    int32_t exact_occupancy;        /* debug: always take the per-agent sequential occupancy filter    */
    int32_t brute_force_scan;       /* debug / A-B: evaluate every (agent, cell) pair in the grid scan    */
    int32_t debug_flags;            /* debug / tests: bit 0 = always evaluate the reward's psi sums in fp64 (skip the fp32 estimate) */
    int32_t obs_layout;             /* SWARM_OBS_REFERENCE: obs [E][obs_dim][n_a] (CPP:324-328, what env.step returns);
                                       SWARM_OBS_AGENT_MAJOR: obs [E][n_a][obs_dim], one contiguous row per agent — for consumers on
                                       the device (swarm_policy_step with obs_agent_major, a replay ring slot); same values    */
    int32_t variant;                /* SWARM_VARIANT_ASSEMBLY (the reference env) or SWARM_VARIANT_FLOCKING (VARIANTS.md 3)      */
    double d_sen;                   /* 0.4                                             ENV:199          */
    double r_avoid;                 /*                                                 ENV:124          */
    double size_a;                  /* 0.035                                           ENV:44           */
    double k_ball, k_wall, c_wall;  /* 30, 100, 5                                      ENV:71,73,74     */
    double dt, vel_max, mass;       /* 0.1, 0.8, 1                                     ENV:79,52,40     */
    double boundary_pos[4];         /* xmin, ymax, xmax, ymin                          ENV:193-196      */
} swarm_config;

/* Device buffers owned by the CALLER (e.g. torch tensors); every pointer is a device pointer on
 * `config.device` and must stay valid for the life of the handle.  OUT = f64 or f32 per out_dtype. */
typedef struct swarm_buffers {
    int32_t struct_size;
    int32_t pad_;
    double *p;                 /* [E][2][n_a]            in/out   ENV:203-208 */
    double *dp;                /* [E][2][n_a]            in/out   ENV:215     */
    double *grid;              /* [E][n_g_pad][2]        internal cell-major copy of grid_center, written by
                                  swarm_set_grid; n_g_pad = swarm_grid_pad(n_g_max)                      */
    int32_t *n_g;              /* [E]                    written by swarm_set_grid                         */
    float *word_box;           /* [E][n_g_pad/32][4]     written by swarm_set_grid: bounding box of every 32-cell word    */
    double *frame;             /* [E][2]                 written by swarm_set_grid: unit axis of the env's box frame      */
    double *in_thresh;         /* [E]                    written by swarm_set_grid (in-shape threshold)    */
    void *obs;                 /* [E][obs_dim][n_a] OUT  ENV:227, layout CPP:324-328                       */
    void *reward;              /* [E][1][n_a]       OUT  ENV:353                                           */
    void *a_prior[2];          /* 2 x [E][2][n_a]   OUT  ENV:612; double-buffered, see swarm_a_prior_ptr   */
    int32_t *neighbor_index;   /* [E][n_a][6]            ENV:228                                           */
    int32_t *in_flags;         /* [E][n_a]               ENV:229                                           */
    int32_t *nearest_cell;     /* [E][n_a]               index of the nearest cell (CPP:884-885); also the seed of the
                                                         next step's nearest-cell search (any content is a valid seed) */
    int32_t *sensed_index;     /* [E][n_a][80]           ENV:230   (may be NULL unless emit_indices)       */
    int32_t *occupied_index;   /* [E][n_a][200]          ENV:231   (may be NULL unless emit_indices)       */
} swarm_buffers;

/* cells per env rounded up to the kernel's tile (multiple of 32) */
int32_t swarm_grid_pad(int32_t n_g_max);
/* 2*2*(6+1+self)+2*80, ENV:801 */
int32_t swarm_obs_dim(const swarm_config *cfg);

int swarm_create(const swarm_config *cfg, const swarm_buffers *buf, swarm_sim **out);
int swarm_destroy(swarm_sim *sim);

/* Upload target shapes for envs [env0, env0+count).  grid: per env a block of 2*n_g_max doubles whose first
 * 2*n_g[e] hold the reference's grid_center[2][n_g] (ENV:187) — host pointer unless grid_on_device != 0.
 * n_g, l_cell: host arrays [count] (ENV:163,179).  Invalidates the cached prior (like eval_assembly.py:34-57
 * poking env.grid_center between steps). */
int swarm_set_grid(swarm_sim *sim, int32_t env0, int32_t count, const double *grid, int grid_on_device,
                   const int32_t *n_g, const double *l_cell, void *stream);

/* Device-resident shape library for swarm_reset(): n_shapes blocks of 2*n_g_max doubles (host), each holding a shape's
 * origin-frame grid [2][n_g] (the transposed `grid_coords` of the reference's results.pkl, ENV:117,164), with its cell
 * count and cell size (ENV:116,163). */
int swarm_set_shapes(swarm_sim *sim, int32_t n_shapes, const double *grids, const int32_t *n_g, const double *l_cell);

/* Target shapes for envs [env0, env0+count) as (library shape, pose) pairs chosen by the host: the device computes
 * grid_center = R * origin + off itself, R = [[cos, sin], [-sin, cos]], every product and sum rounded separately (ENV:175-187
 * evaluated without FMA).  shape_ids: HOST [count]; pose: HOST [count][4] = (cos, sin, off_x, off_y).  Same effect as
 * swarm_set_grid with that grid, and the pose is known exactly (swarm_fast_path may then return 2). */
int swarm_set_grid_pose(swarm_sim *sim, int32_t env0, int32_t count, const int32_t *shape_ids, const double *pose, void *stream);

/* != 0 if the next step / observe runs the lookup-scan kernel: a shape library was set, the configuration is eligible (single-warp
 * envs, <= 1023 cells, d_sen / l_cell <= 14.9, lattice shapes) and EVERY env's current grid was recognised as a rigid transform
 * of a library shape (swarm_set_grid checks each grid against the library to 1e-9; swarm_reset knows the pose).  Otherwise the
 * general culled scan runs; results are identical either way.  2 = in addition every pose is known exactly (the device built
 * the grids itself: swarm_reset), so the kernel recomputes the cells it needs from the library instead of reading each env's
 * stored copy. */
int swarm_fast_path(const swarm_sim *sim);

/* reset() on the device, ENV:156-223: shape pick, rotation, offset, initial positions and velocities for every env (or
 * those with env_mask[e] != 0; device pointer or NULL), then the observation of the new state (ENV:221).  Random draws come
 * from a counter-based generator keyed by (seed, episode, env_offset + e), not from NumPy's global stream; the map from the
 * draws to grid_center / p / dp is the reference's.  info_dev (device, [E][8] f64, may be NULL) receives per env
 * {shape index, cos, sin, offset_x, offset_y, wide-spawn flag, cluster_centre_x, cluster_centre_y}.  Draw k of env e is
 * u = (mix64(seed, episode, env_offset + e, k) >> 11) * 2^-53 (see k_reset); agent i uses draws 16 + i, 16 + n_a + i (position)
 * and 16 + 2 n_a + i, 16 + 3 n_a + i (velocity), so a host can rebuild p / dp exactly. */
int swarm_reset(swarm_sim *sim, uint64_t seed, uint64_t episode, uint64_t env_offset, const uint8_t *env_mask,
                double *info_dev, void *stream);

/* The same reset for a LIST of envs (device int32 array of `count` distinct env ids): only those envs are re-randomised and
 * re-observed, one CTA each — the auto-reset of a vector env whose episodes end at different steps (ENV:156-223 per env). */
int swarm_reset_envs(swarm_sim *sim, uint64_t seed, uint64_t episode, uint64_t env_offset, const int32_t *env_list_dev,
                     int32_t count, double *info_dev, void *stream);

/* Measurement aid (bench.py): dense FMA throughput of `device` in TFLOP/s, fp32 and fp64, from a register-resident FMA loop —
 * the roofline denominator of the O(n_a^2) large-swarm configuration (SURVEY.md 8(d)). */
int swarm_measure_fma_peak(int32_t device, double *fp32_tflops, double *fp64_tflops);

/* Self-test (tests only): the prior's shared-reciprocal division against the correctly rounded a / b on n pseudo-random operand
 * pairs; kind 0 = simulator magnitudes, 1 = wide exponents, 2 = divisors 1..6.  *mismatches must come back 0. */
int swarm_selftest_division(int32_t device, uint64_t n, uint64_t seed, int32_t kind, uint64_t *mismatches);

/* Evaluation metrics of the reference wrapper for every env, on the device: out_dev [E][3] f64 =
 * {coverage_rate, distribution_uniformity, voronoi_based_uniformity} (assembly_wrapper.py:48-72, 74-101, 103-129). */
int swarm_metrics(swarm_sim *sim, double *out_dev, void *stream);

/* ---- Rendering: rgb_array frames (gym's layout, uint8 [count][height][width][3]) of any set of envs, on the device.
 * Pixel rules, all fp64 with every operation rounded separately (the library is built with -fmad=false):
 *   view (x0, y1, x1, y0) = (xmin, ymax, xmax, ymin); sx = (x1 - x0) / W, sy = (y1 - y0) / H; the centre of pixel (row r, col c)
 *   is X = x0 + (c + 0.5) * sx, Y = y1 - (r + 0.5) * sy (row 0 = top).  A disc (cx, cy, rr) covers it iff dx*dx + dy*dy <= rr,
 *   dx = X - cx, dy = Y - cy, evaluated dx*dx, then dy*dy, then the sum.  Layers, bottom to top (the topmost covering one decides):
 *   1. background: SWARM_RGB_ARENA if x_min <= X <= x_max && y_min <= Y <= y_max (the handle's boundary_pos), else SWARM_RGB_OUTSIDE;
 *   2. SWARM_RENDER_CELLS: a disc at every cell j < n_g[e] with rr = in_thresh[e] * 0.5 (the in-shape radius), SWARM_RGB_CELL;
 *   3. SWARM_RENDER_TRAILS: per agent a capsule around each segment A -> B of consecutive trail samples, half-width w = size_a * 0.25:
 *      u = B - A, ll = ux*ux + uy*uy, t = ll > 0 ? ((X - Ax)*ux + (Y - Ay)*uy) / ll : 0 clamped to [0, 1], q = A + t*u, covered iff
 *      (X - qx)^2 + (Y - qy)^2 <= w*w; a segment with |ux| > half_w or |uy| > half_h (a periodic wrap) is not drawn; SWARM_RGB_TRAIL;
 *   4. SWARM_RENDER_AGENTS: a disc at p[e][:, i] with rr = size_a * size_a, SWARM_RGB_AGENT_IN if in_flags[e][i] & 1 (the last
 *      observation) else SWARM_RGB_AGENT_OUT; where several agents cover a pixel the largest index wins.
 * No anti-aliasing.  A flocking handle has no cells, and its agents all take SWARM_RGB_AGENT_OUT. */
#define SWARM_RENDER_CELLS 1
#define SWARM_RENDER_AGENTS 2
#define SWARM_RENDER_TRAILS 4
/* the palette, in this order (R, G, B) */
#define SWARM_RGB_ARENA 255, 255, 255
#define SWARM_RGB_OUTSIDE 160, 160, 160
#define SWARM_RGB_CELL 190, 215, 240
#define SWARM_RGB_TRAIL 250, 170, 90
#define SWARM_RGB_AGENT_IN 40, 150, 40
#define SWARM_RGB_AGENT_OUT 210, 40, 40
typedef struct swarm_render_args {
    int32_t struct_size;               /* sizeof(swarm_render_args)                                                    */
    int32_t width, height;             /* pixels, each in [1, 8192]                                                      */
    int32_t flags;                     /* SWARM_RENDER_* bits                                                            */
    int32_t count;                     /* frames, >= 1                                                                   */
    int32_t pad_;
    const int32_t *env_ids;            /* HOST [count], each in [0, E); duplicates allowed                               */
    double view[4];                    /* xmin, ymax, xmax, ymin (finite, xmin < xmax, ymin < ymax); all zero = the arena  */
    const double *trail;               /* DEVICE ring [trail_cap][count][2][n_a] f64 of past positions, or NULL          */
    int32_t trail_cap, trail_len;      /* 0 <= trail_len <= trail_cap <= 1024: the trail_len newest samples are drawn     */
    int32_t trail_head;                /* ring slot of the newest sample, in [0, trail_cap) when trail_len > 0           */
    int32_t pad2_;
    uint8_t *frames;                   /* DEVICE [count][height][width][3]                                               */
} swarm_render_args;
/* Draws frame f of env env_ids[f] from the handle's current p, in_flags and cells.  Every argument is checked before anything is
 * launched (SWARM_ERR_INVALID, frames untouched).  Stream-ordered, no host synchronisation; one launch per 2048 frames, counted in
 * swarm_launch_count. */
int swarm_render(swarm_sim *sim, const swarm_render_args *args, void *stream);
/* Copies the palette (6 RGB triples in the order of the SWARM_RGB_* macros above) to rgb[18] unless NULL; returns 6. */
int swarm_render_palette(uint8_t *rgb);

/* The reference env's own action strategies (ENV:519-601, Python/NumPy there) for the CURRENT state of every env:
 * SWARM_STRATEGY_RULE = agent_strategy 'rule' (ENV:530-601, the expert controller of collect_expert_data.py),
 * SWARM_STRATEGY_LLM = 'llm' (ENV:524-529 -> robot_prior_policy ENV:876-941; uses the neighbour list of the last
 * observation).  act_dev: DEVICE [E][2][n_a] f64, to be passed to swarm_step with SWARM_F64 (ENV:633 u = a).
 * Arithmetic: plain IEEE binary64 in the reference's evaluation order; the NumPy original itself varies in the last
 * bits with the NumPy / BLAS build (np.linalg.norm -> BLAS dot, pairwise np.sum), agreement is ~1e-15. */
#define SWARM_STRATEGY_RULE 1
#define SWARM_STRATEGY_LLM 2
int swarm_strategy_actions(swarm_sim *sim, int kind, double *act_dev, void *stream);

/* Redirect the observation output of the following observe / step calls to another device buffer of the same shape and
 * dtype.  Lets a device-resident rollout loop keep the previous observation (policy input, replay `obs`) and the new one
 * (replay `next_obs`) without a copy: alternate two buffers. */
int swarm_set_obs_buffer(swarm_sim *sim, void *obs_dev);

/* Tell the handle that the caller overwrote p / dp (device buffers) outside step(): the next step recomputes the
 * prior from the new state and the stale neighbor_index, exactly like the reference would (ENV:613-624). */
int swarm_mark_state_dirty(swarm_sim *sim);

/* State restore (checkpoint / handle rebuilt with a larger n_g_max): the caller copied neighbor_index, in_flags and
 * nearest_cell (and whatever outputs it wants to keep) of an earlier observation into this handle's buffers; the handle
 * treats them as its last observation, so swarm_step is legal and computes its prior from that neighbour list
 * (ENV:613-624 uses the neighbor_index of the last _get_obs call).  swarm_is_observed: 1 once an observation exists. */
int swarm_restore_observation(swarm_sim *sim);
int swarm_is_observed(const swarm_sim *sim);

/* ---- FlockingSwarm variant (VARIANTS.md 3).  The reference registers `FlockingSwarm-v0` (cus_gym/gym/envs/__init__.py:7-12) but
 * ships no source for it, so this is a SPECIFIED variant with no oracle (parity unpinned).  A handle created with
 * variant = SWARM_VARIANT_FLOCKING (n_a <= 128) has obs [E][4 * (6 + is_con_self_state)][n_a] = the assembly observation's head rows
 * (CPP:102-126); the grid buffers are unused (tiny dummies are fine).  swarm_flock_step = the assembly step's pair phase, walls /
 * periodic wrap, integrator, k-NN and head rows (the SAME first-half kernel, ENV:442-457, 631-652, CPP:628-698, 775-807, 835-846)
 * followed by the Reynolds reward of VARIANTS.md 3 into `reward` of the handle; swarm_flock_observe = the same without dynamics. */
int swarm_flock_observe(swarm_sim *sim, void *stream);
int swarm_flock_step(swarm_sim *sim, const void *act, int act_dtype, void *stream);

/* ---- PredatorPreySwarm variant (VARIANTS.md 4).  Registered by the reference (cus_gym/gym/envs/__init__.py:14-19), no source
 * shipped: a SPECIFIED variant, parity unpinned.  Stateless calls: the caller owns every buffer (device memory).  Agents
 * [0, n_p) are pursuers, [n_p, n_p + n_e) escapers, n_p + n_e <= 128.  obs [E][4 * (12 + is_con_self_state)][n]: the assembly head
 * rows (CPP:102-126) over the 6 nearest agents of the own type, then of the other type; neighbor_index [E][n][12] likewise. */
enum { SWARM_PP_INPUT = 0, SWARM_PP_STATIC = 1, SWARM_PP_RANDOM = 2, SWARM_PP_NEAREST = 3 };
typedef struct swarm_pp_config {
    uint32_t struct_size;
    int32_t device, num_envs, n_p, n_e;
    int32_t is_con_self_state, is_periodic, billiards;   /* billiards: elastic walls instead of the wall spring / damper         */
    int32_t out_dtype;                                   /* SWARM_F32 / SWARM_F64 for obs and reward                             */
    int32_t strategy_p, strategy_e;                      /* SWARM_PP_*: whose actions come from `act`, who is scripted           */
    double d_sen, size_a, k_ball, k_wall, c_wall, dt, vel_max_p, vel_max_e, mass;
    double boundary_pos[4];                              /* x_min, y_max, x_max, y_min like ENV:117                              */
    uint64_t seed;                                       /* SWARM_PP_RANDOM draws: counter-based on (seed, step_index, env, agent) */
} swarm_pp_config;
typedef struct swarm_pp_buffers {
    uint32_t struct_size;
    double *p, *dp;                 /* [E][2][n] f64, updated in place by swarm_pp_step                                          */
    void *obs, *reward;             /* [E][obs_dim][n], [E][n] in out_dtype                                                      */
    int32_t *neighbor_index;        /* [E][n][12]                                                                                */
} swarm_pp_buffers;
int swarm_pp_obs_dim(const swarm_pp_config *cfg);
int swarm_pp_observe(const swarm_pp_config *cfg, const swarm_pp_buffers *buf, void *stream);
int swarm_pp_step(const swarm_pp_config *cfg, const swarm_pp_buffers *buf, const void *act, int act_dtype, uint64_t step_index,
                  void *stream);

/* reset() tail, ENV:221 -> _get_obs: observation (+ reward) of the current state, no dynamics. */
int swarm_observe(swarm_sim *sim, void *stream);

/* env.step(a), ENV:487-666 (agent_strategy 'input', Cartesian).  act: DEVICE [E][2][n_a], f32 or f64. */
int swarm_step(swarm_sim *sim, const void *act, int act_dtype, void *stream);

/* Same step through HOST buffers (pinned or pageable): H2D act, step, D2H obs / reward / a_prior (NULL = skip),
 * synchronises the stream before returning.  This is the call a host-side caller of the reference would make. */
int swarm_step_host(swarm_sim *sim, const float *act_host, void *obs_host, void *reward_host, void *a_prior_host,
                    void *stream);

/* a_prior returned by the most recent swarm_step (the reference's 5th return value, ENV:666). */
void *swarm_a_prior_ptr(swarm_sim *sim);

/* Synthetic actions U(-1,1) f32 [E][2][n_a] from a counter-based generator keyed by (seed, step, env_offset+e, k);
 * bit-identical to oracle/assembly_oracle.c:orc_fill_actions.  Benchmark / test input only. */
int swarm_fill_actions(swarm_sim *sim, uint64_t seed, uint64_t step, uint64_t env_offset, float *act_dev, void *stream);

/* Test hook: psi = _rho_cos_dec(z, delta = 0, r) (CPP:1012-1020) of n HOST values through the device implementation
 * (the kernels use their own [0, pi] cosine instead of libdevice's). */
int swarm_debug_rho(const double *z_host, int32_t n, double r, double *out_host);

/* number of kernels this handle has launched so far */
int64_t swarm_launch_count(const swarm_sim *sim);
/* dynamic shared memory bytes and threads per CTA of the fused step kernel for this handle */
int swarm_kernel_geometry(const swarm_sim *sim, int32_t *threads_per_cta, int32_t *smem_bytes, int32_t *ctas);

/* Host-only helper (no GPU needed), exposed for tests: the double T with  sqrt(s) < d  <=>  s < T  (le == 0), or the
 * double U with  sqrt(s) <= d  <=>  s <= U  (le != 0), sqrt being IEEE round-to-nearest.  The kernels compare squared
 * distances with these instead of taking square roots. */
double swarm_sqrt_threshold(double d, int le);

/* ============================================================================================
 * (3) Device-resident replay storage (SURVEY.md §8 f1) — replaces the host NumPy ring of
 *     marl_llm/algorithm/utils/buffer_agent.py (= BUF) for the batched simulator.  Stateless: the caller owns the ring
 *     arrays (device, f32, row-major [capacity][dim]) and the write cursor; the host mirror
 *     (marl_llm_b200/rollout.py:ReplayBufferAgent) keeps curr_i / filled_i exactly like BUF:96-127.
 * ============================================================================================ */
typedef struct swarm_rollout_buffers {
    int32_t struct_size, obs_dim, act_dim, pad_;
    int64_t capacity;                 /* rows = max_steps * num_agents (BUF:46) */
    float *obs, *act, *act_prior, *log_pi, *rew, *next_obs, *done;   /* BUF:49-55; act_prior / log_pi may be NULL */
} swarm_rollout_buffers;

/* push(), BUF:67-128, for num_envs envs at once: the simulator's feature-major arrays (obs / next_obs [E][obs_dim][n_a],
 * reward [E][1][n_a], act_prior [E][act_dim][n_a] in out_dtype; act [E][act_dim][n_a] in act_dtype; done [E][1][n_a] bool;
 * log_pi [E][1][n_a] f32 or NULL) are transposed to agent rows (BUF:86-90, agents [agent_start, agent_stop) of every env,
 * env-major) and written to ring rows [row0, row0 + E*(agent_stop-agent_start)). */
int swarm_rollout_push(const swarm_rollout_buffers *buf, int64_t row0, int32_t num_envs, int32_t n_a, int32_t agent_start,
                       int32_t agent_stop, const void *obs, const void *next_obs, const void *reward, const uint8_t *done,
                       const void *act_prior, int out_dtype, const void *act, int act_dtype, const float *log_pi, void *stream);

/* The same push in parts (SWARM_PUSH_* bit mask): lets a time-indexed ring (obs of step t+1 = next_obs of step t, one
 * array) store each observation once — SWARM_PUSH_OBS alone transposes `obs` into ring rows [row0, ...), SWARM_PUSH_SMALL
 * alone writes act / act_prior / reward / done / log_pi.  Inputs of parts that are not requested may be NULL. */
#define SWARM_PUSH_OBS 1
#define SWARM_PUSH_NEXT_OBS 2
#define SWARM_PUSH_SMALL 4
int swarm_rollout_push_parts(const swarm_rollout_buffers *buf, int64_t row0, int32_t num_envs, int32_t n_a, int32_t agent_start,
                             int32_t agent_stop, const void *obs, const void *next_obs, const void *reward, const uint8_t *done,
                             const void *act_prior, int out_dtype, const void *act, int act_dtype, const float *log_pi, int parts,
                             void *stream);

/* the gather of sample(), BUF:152-161: rows_dev [n] int64 ring rows (device) -> [n][dim] f32 outputs (device);
 * act_prior / log_pi outputs may be NULL (BUF:159-162 is_prior / is_log_pi). */
int swarm_rollout_gather(const swarm_rollout_buffers *buf, const int64_t *rows_dev, int32_t n, float *obs, float *act, float *reward,
                         float *next_obs, float *done, float *act_prior, float *log_pi, void *stream);

/* ============================================================================================
 * (4) Rollout policy on the device (SURVEY.md §8 f1): MADDPG.step() of marl_llm/algorithm/algorithms/maddpg.py:72-87
 *     (DDPGAgent.step, utils/agents.py:69-96; MLPNetwork.forward, utils/networks.py:33-44) for every agent of every env,
 *     reading the simulator's obs layout and writing its action layout.  fp32 FFMA, fp32 accumulation.
 * ============================================================================================ */
typedef struct swarm_policy swarm_policy;

/* obs_dim, hidden_dim <= 192 (reference: 192, 180), act_dim <= 8 (reference: 2). */
int swarm_policy_create(int32_t device, int32_t obs_dim, int32_t hidden_dim, int32_t act_dim, swarm_policy **out);
int swarm_policy_destroy(swarm_policy *p);
/* HOST pointers, torch nn.Linear layout: w1 [hidden][obs_dim], w2, w3 [hidden][hidden], w4 [act_dim][hidden], biases [out]
 * (networks.py:22-25 fc1..fc4). */
int swarm_policy_load(swarm_policy *p, const float *w1, const float *b1, const float *w2, const float *b2, const float *w3,
                      const float *b3, const float *w4, const float *b4);
/* obs: DEVICE [E][obs_dim][n_a] f32 -> act: DEVICE [E][act_dim][n_a] f32 = tanh(fc4(lrelu(fc3(lrelu(fc2(lrelu(fc1 obs))))))).
 * explore (agents.py:85-93): 0 none; 1 act += noise_scale * N(0,1), clamp to [-1,1]; 2 act = U(-1,1) (the epsilon branch; the
 * caller draws epsilon once per step like the reference).  Noise comes from a counter-based generator keyed by
 * (seed, step, column, component), not from NumPy.  log_pi: DEVICE [E][1][n_a] f32 or NULL (agents.py:82,88,91). */
int swarm_policy_step(swarm_policy *p, const float *obs, int32_t num_envs, int32_t n_a, float *act, float *log_pi, int explore,
                      float noise_scale, uint64_t seed, uint64_t step, void *stream);
/* Arithmetic of swarm_policy_step.  SWARM_POLICY_FP32 (default): fp32 FFMA, agrees with torch's fp32 network to rounding.
 * SWARM_POLICY_F16_TC: one persistent tcgen05 kernel (weights resident in shared memory as fp16, activations and fp32
 * accumulators in tensor memory); ~50x faster, deviates by ~1e-3 absolute on the tanh output. */
#define SWARM_POLICY_FP32 0
#define SWARM_POLICY_F16_TC 1
/* SWARM_POLICY_F16X3_TC: fp32-accurate tensor-core path: every operand is split into two fp16 numbers (hi + lo, 22 bits),
 * three tcgen05.mma per k-step (hi*hi + lo*hi + hi*lo) into one fp32 accumulator, weights streamed through a 3-slot
 * shared-memory ring.  Agrees with the fp32 network to ~1e-6 (|values| must stay below 65504). */
#define SWARM_POLICY_F16X3_TC 2
int swarm_policy_set_precision(swarm_policy *p, int precision);
/* test hook: when non-NULL, the tensor-core path also writes its layer-1 accumulators (fc1 without bias) to
 * layer1_acc_dev [E*n_a][192] f32 (device). */
int swarm_policy_debug_buffer(swarm_policy *p, float *layer1_acc_dev);
int64_t swarm_policy_launch_count(const swarm_policy *p);

/* gather for a time-indexed ring: next_obs of ring row r is row r + next_row_offset of the OBS array (buf->next_obs may be
 * NULL); next_row_offset < 0 behaves like swarm_rollout_gather.  Precondition for both gathers: 0 <= rows[k] and
 * rows[k] + max(next_row_offset, 0) < buf->capacity; a row outside that range is clamped into it by the kernel (never read
 * out of bounds), so validate indices on the host if a wrong index must be an error. */
int swarm_rollout_gather_ring(const swarm_rollout_buffers *buf, const int64_t *rows_dev, int32_t n, int64_t next_row_offset, float *obs,
                              float *act, float *reward, float *next_obs, float *done, float *act_prior, float *log_pi, void *stream);

/* While non-NULL, swarm_policy_step also writes every agent's observation as one fp32 row, rows_dev [E*n_a][obs_dim] (device):
 * the transposition a replay push would do, for free, from the registers of the threads that read the observation anyway. */
int swarm_policy_rows_out(swarm_policy *p, float *rows_dev);

/* agent_major != 0: the obs pointer of the following swarm_policy_step calls is agent-major, [E*n_a][obs_dim] — the output of a
 * simulator created with SWARM_OBS_AGENT_MAJOR (each loader thread then reads 128 contiguous bytes instead of 32 strided words),
 * e.g. a slot of a time-indexed replay ring the simulator wrote its observation into directly. */
int swarm_policy_obs_layout(swarm_policy *p, int agent_major);

/* ============================================================================================
 * (5) State store: save env states of a batched handle on the device and load them back into the same or another handle,
 *     one state into many envs (clone = save + load with a repeated slot).  Every step after a load is bit-identical to the
 *     run the saved envs would have continued (DESIGN.md §11).
 * ============================================================================================ */
typedef struct swarm_state_store swarm_state_store;   /* opaque, library-owned device memory on the handle's device */

/* `capacity` slots, each holding one env's complete state, for handles of sim's configuration: every field of swarm_config
 * except num_envs, the device included.  Flocking handles: SWARM_ERR_UNSUPPORTED.  The store has its own lifetime. */
int swarm_state_store_create(const swarm_sim *sim, int64_t capacity, swarm_state_store **out);
int swarm_state_store_destroy(swarm_state_store *st);
/* bytes of one slot (the layout is private to the library); 0 when st is NULL */
int64_t swarm_state_slot_bytes(const swarm_state_store *st);
/* A slot holds p, dp, the padded grid row, word_box, frame, n_g, in_thresh, the library pose and shape id, nearest_cell,
 * neighbor_index, in_flags, obs (of the current observation buffer), reward; with want_prior the prior of the current state and
 * the prior the last step returned; with emit_indices sensed_index and occupied_index (done is constant).  The store also keeps,
 * per slot on the host, the source env's match record, whether the source's prior was valid and the fingerprint of the source's
 * shape library.
 *
 * swarm_state_save: slot slots[k] <- env env_ids[k] of sim.  env_ids, slots: HOST [count]; slots distinct; sim observed.
 * swarm_state_load: env env_ids[k] of sim <- slot slots[k].  env_ids distinct, slots filled and may repeat.  sim may be any handle
 * of the store's configuration; one that was never observed only when env_ids covers every env (it is observed afterwards).
 * A slot saved under another shape library (swarm_set_shapes) is restored as unmatched: the general scan serves that env, with the
 * same results.  A slot whose prior was stale (state changed behind the handle's back) makes the next step recompute the prior.
 * Every argument is checked before anything is launched (SWARM_ERR_INVALID; handle and store unchanged).  Stream-ordered, no host
 * synchronisation and no host-to-device copy: the pairs travel in the kernel parameters (one launch per 2048 pairs, counted in
 * sim's swarm_launch_count); the caller may free the host arrays when the call returns. */
int swarm_state_save(swarm_sim *sim, swarm_state_store *st, const int32_t *env_ids, const int32_t *slots, int32_t count, void *stream);
int swarm_state_load(swarm_sim *sim, swarm_state_store *st, const int32_t *slots, const int32_t *env_ids, int32_t count, void *stream);

/* ============================================================================================
 * (6) Prior policies as programs (DESIGN.md §12).  A caller's `robot_policy` (include/swarm_prior_api.cuh, which states the
 *     contract) is compiled at run time into an sm_100a CUBIN and runs as the step's prior (a_prior) or as actions.
 * ============================================================================================ */
typedef struct swarm_prior_program swarm_prior_program;   /* opaque: a loaded CUBIN on one device */
typedef struct swarm_prior_population swarm_prior_population;   /* opaque: programs and an assignment env -> program */

/* Host only, no GPU needed: source -> sm_100a CUBIN.  The library appends the entry points of swarm_prior_api.cuh (whose text it
 * embeds) and compiles with its fixed options --gpu-architecture=sm_100a --fmad=false -default-device (IEEE division and square
 * root).  NVRTC is opened with dlopen on the first call: nvrtc_path, or libnvrtc.so.12 on the loader path when it is NULL; not
 * found: SWARM_ERR_UNSUPPORTED, naming the path tried.  Two-call size query: with image = NULL only *image_size is written; then
 * image_cap >= *image_size bytes at image.  NVRTC's log (errors with their line, warnings) goes to log[log_cap], NUL-terminated
 * and truncated, when log is non-NULL.  A source that does not compile, or has no robot_policy: SWARM_ERR_INVALID. */
int swarm_prior_compile(const char *source, const char *nvrtc_path, void *image, int64_t image_cap, int64_t *image_size, char *log,
                        int64_t log_cap);
/* Loads a CUBIN of swarm_prior_compile on `device` (cudaLibraryLoadData: no driver JIT).  Programs and populations are owned by
 * the caller: destroy a program only after it is removed from every handle it is installed on and every population that lists it
 * is destroyed, and a population only after it is removed from every handle it is installed on. */
int swarm_prior_program_create(int32_t device, const void *image, int64_t size, swarm_prior_program **out);
int swarm_prior_program_destroy(swarm_prior_program *prog);
/* Installs prog as sim's prior: every following swarm_step launches prog's a_prior entry (in the handle's output dtype) on the
 * pre-step state before the step kernel, which then skips its own prior, and swarm_observe writes no prior.  The nearest cell a
 * program sees is the one the last observation stored while that observation is of the current state and grid, else it is
 * scanned.  prog = NULL: the built-in prior again, from the next step on.  Needs want_prior (else SWARM_ERR_INVALID) and an
 * assembly handle (flocking: SWARM_ERR_UNSUPPORTED); prog on sim's device.  While a program is installed, swarm_state_save records
 * the slots' prior as stale, so a load into any handle recomputes it. */
int swarm_set_prior_program(swarm_sim *sim, swarm_prior_program *prog);
/* prog as the controller (the 'llm' strategy's use of the prior): act_dev [E][2][n_a] f64 (device) from the current state and
 * the neighbour list of the last observation (sim must be observed).  Legal whether or not sim has want_prior. */
int swarm_prior_program_actions(swarm_sim *sim, swarm_prior_program *prog, double *act_dev, void *stream);
/* A population: `count` programs and the program env_program[e] (HOST [num_envs], values in [0, count)) of every env of a handle
 * with num_envs envs.  Each program runs on its own envs only, so K candidate priors share one batch and one step.  The envs are
 * grouped by program (ascending env id within a group) and the list is copied once to device memory the population owns (a
 * synchronous copy).  A program without envs is allowed; it launches nothing.  Checked before anything is allocated
 * (SWARM_ERR_INVALID, nothing created): count >= 1, num_envs >= 1, no NULL program, every program on `device`, every
 * env_program[e] in range.  The caller may free both host arrays when the call returns. */
int swarm_prior_population_create(int32_t device, int32_t num_envs, int32_t count, swarm_prior_program *const *programs,
                                  const int32_t *env_program, swarm_prior_population **out);
int swarm_prior_population_destroy(swarm_prior_population *pop);
/* Installs pop as sim's prior: every following swarm_step launches, in program order, each program's a_prior entry (in the
 * handle's output dtype) over that program's envs, one launch per program with envs (counted in swarm_launch_count), then the
 * step kernel without its own prior; otherwise as swarm_set_prior_program.  Installing a population replaces an installed
 * program, and installing a program replaces a population.  pop = NULL: the built-in prior again, from the next step on.  Needs
 * want_prior (else SWARM_ERR_INVALID) and an assembly handle (flocking: SWARM_ERR_UNSUPPORTED); pop on sim's device and made for
 * sim's num_envs (else SWARM_ERR_INVALID).  A rejected call leaves the installed prior in force. */
int swarm_set_prior_population(swarm_sim *sim, swarm_prior_population *pop);
/* Every env's program as the controller: act_dev [E][2][n_a] f64 (device), each env's rows written by its program, from the
 * current state and the neighbour list of the last observation (sim must be observed; pop made for sim's device and num_envs).
 * Legal whether or not sim has want_prior. */
int swarm_prior_population_actions(swarm_sim *sim, swarm_prior_population *pop, double *act_dev, void *stream);

const char *swarm_last_error(void);
int swarm_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SWARM_B200_H */
