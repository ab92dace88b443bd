// swarm_abi.cu — host side of the C ABI declared in include/swarm_b200.h.
//
// There is no CPU implementation behind these entry points: without a usable sm_100 device the batched calls
// return SWARM_ERR_NO_DEVICE / SWARM_ERR_CUDA and the legacy (void) calls print the CUDA error and abort.
#include "swarm_kernels.cuh"
#include "render_kernels.cuh"
#include "state_kernels.cuh"
#include "../../include/swarm_b200.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

using namespace swarm;

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string &msg) { g_last_error = msg; return code; }

#define CU_TRY(expr)                                                                                   \
    do {                                                                                               \
        cudaError_t err__ = (expr);                                                                    \
        if (err__ != cudaSuccess)                                                                      \
            return fail(SWARM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(err__));        \
    } while (0)

// smallest double T with sqrt_rn(T) >= d, i.e.  sqrt_rn(s) < d  <=>  s < T   (sqrt_rn is monotone)
double thresh_lt(double d) {
    if (!(d > 0)) return 0.0;
    double t = d * d;
    while (std::sqrt(t) >= d) t = std::nextafter(t, -INFINITY);
    while (std::sqrt(std::nextafter(t, INFINITY)) < d) t = std::nextafter(t, INFINITY);
    return std::nextafter(t, INFINITY);
}
// largest double U with sqrt_rn(U) <= h, i.e.  sqrt_rn(s) <= h  <=>  s <= U
double thresh_le(double h) {
    if (h < 0) return -1.0;
    double t = h * h;
    while (std::sqrt(t) > h) t = std::nextafter(t, -INFINITY);
    while (std::sqrt(std::nextafter(t, INFINITY)) <= h) t = std::nextafter(t, INFINITY);
    return t;
}

int round32(int n) { return (n + 31) & ~31; }

size_t step_smem_bytes(int nt, int n_words, bool emit, int n_obs, int phase = 0, int rec_cap = -1, int lat_n = 0) {
    if (phase == 1)      // first half: state tile + 2 mbarrier slots (unused) + neighbour list + filter positions (k_step: SLIM)
        return (size_t)4 * nt * sizeof(double) + 16 + (size_t)TOPO * nt * sizeof(int) + (size_t)nt * sizeof(float2);
    size_t ring = (size_t)2 * CHUNK_CELLS * sizeof(double2);
    if (rec_cap >= 0) ring = std::max(ring, (size_t)(nt / 32) * ((size_t)4 * rec_cap + 128 + 16));      // lookup scan: per warp, row records + running counts
    size_t b = ring + (rec_cap >= 0 ? 0 : (size_t)n_words * sizeof(float4)) + (size_t)4 * nt * sizeof(double);   // TMA ring / records + word boxes + state tile
    b += (size_t)n_words * nt * 4 * (emit ? 2 : 1);
    b += (size_t)((n_words + 3) & ~3) * 4 + 16;                                                    // covered mask + 2 mbarriers
    if (phase != 2) {                                                                                // the second-half kernel parks its neighbour list on the idle ring
        b += (size_t)TOPO * nt * sizeof(int);                                                       // neighbour list
        b += (size_t)nt * sizeof(float2);                                                            // fp32 positions (pair-loop filter)
    }
    if (rec_cap >= 0) b += (size_t)(3 * lat_n + lat_n / 4) * 8;                                            // lookup scan: lattice tables of the env's shape
    const size_t scratch = (size_t)3 * n_obs * sizeof(double) + 32 * sizeof(int);                   // sparse schedule scratch:
    if (nt == 32 && n_words <= 32 && scratch > ring) b += scratch;   // aliases the TMA ring when it fits
    return b;
}

typedef void (*step_fn_t)(const KParams);

// cudaFuncAttributeMaxDynamicSharedMemorySize is per kernel function and process-wide: several handles (and the legacy entry
// points) share the instantiations, so the attribute is only ever RAISED (a handle with a smaller need must not shrink it)
cudaError_t raise_smem_limit(const void *fn, size_t bytes) {
    static std::mutex mu;
    static std::map<const void *, size_t> high;
    std::lock_guard<std::mutex> lock(mu);
    size_t &h = high[fn];
    if (bytes <= h) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) h = bytes;
    return e;
}

// grows a device staging buffer to hold at least n elements (its contents are not kept)
template <typename T>
int grow_staging(T *&buf, size_t &cap, size_t n) {
    if (n <= cap) return SWARM_OK;
    if (buf) CU_TRY(cudaFree(buf));
    buf = nullptr; cap = 0;
    CU_TRY(cudaMalloc(&buf, n * sizeof(T)));
    cap = n;
    return SWARM_OK;
}

// The k_step instantiations the host launches, by key (template parameters: see k_step).  MAXT 1024 exists for PH 0 only and
// WIDE for PH 1 only.  The first half never writes the index arrays, so it has no EMIT instantiation; the lookup-scan second
// half (PH 2, FAST 1 / 2) exists for DYN = false only.
template <typename OUT, bool DYN, bool EMIT>
step_fn_t step_kernel(int maxt, int ph, int fast, bool wide) {
    if (maxt == 1024)
        return fast == 0 ? (step_fn_t)k_step<OUT, DYN, EMIT, 1024, 0>
             : fast == 1 ? (step_fn_t)k_step<OUT, DYN, EMIT, 1024, 0, 1> : (step_fn_t)k_step<OUT, DYN, EMIT, 1024, 0, 2>;
    if (ph == 0) return k_step<OUT, DYN, EMIT, 128, 0>;
    if (ph == 1) return wide ? (step_fn_t)k_step<OUT, DYN, false, 128, 1, 0, true> : (step_fn_t)k_step<OUT, DYN, false, 128, 1>;
    return fast == 0 ? (step_fn_t)k_step<OUT, DYN, EMIT, 128, 2>
         : fast == 1 ? (step_fn_t)k_step<OUT, false, EMIT, 128, 2, 1> : (step_fn_t)k_step<OUT, false, EMIT, 128, 2, 2>;
}
step_fn_t step_kernel(bool f32, bool dyn, bool emit, int maxt, int ph, int fast = 0, bool wide = false) {
    if (f32) {
        if (dyn) return emit ? step_kernel<float, true, true>(maxt, ph, fast, wide) : step_kernel<float, true, false>(maxt, ph, fast, wide);
        return emit ? step_kernel<float, false, true>(maxt, ph, fast, wide) : step_kernel<float, false, false>(maxt, ph, fast, wide);
    }
    if (dyn) return emit ? step_kernel<double, true, true>(maxt, ph, fast, wide) : step_kernel<double, true, false>(maxt, ph, fast, wide);
    return emit ? step_kernel<double, false, true>(maxt, ph, fast, wide) : step_kernel<double, false, false>(maxt, ph, fast, wide);
}

void fill_constants(KParams &K, int n_a, int n_g_max, int n_obs, int n_occ, bool self_state, bool want_prior,
                    bool exact_occ, bool periodic, double d_sen, double r_avoid, double size_a, double k_ball, double k_wall,
                    double c_wall, double dt, double vel_max, double mass, const double *bp) {
    K.n_a = n_a;
    K.n_g_pad = round32(n_g_max);
    K.n_words = K.n_g_pad / 32;
    K.n_obs_max = n_obs;
    K.n_occ_max = n_occ;
    K.self_state = self_state;
    K.obs_dim = 2 * 2 * (TOPO + 1 + (self_state ? 1 : 0)) + 2 * n_obs;    // ENV:801
    K.want_prior = want_prior;
    K.exact_occ = exact_occ;
    K.periodic = periodic;
    K.half_w = (bp[2] - bp[0]) / 2.0; K.half_h = (bp[1] - bp[3]) / 2.0;      // CPP:70-71
    K.d_sen = d_sen; K.r_avoid = r_avoid; K.size_a = size_a; K.two_size = size_a + size_a;   // ENV:785-786
    K.k_ball = k_ball; K.k_wall = k_wall; K.c_wall = c_wall; K.dt = dt; K.vel_max = vel_max; K.mass = mass;
    K.bx_min = bp[0]; K.by_max = bp[1]; K.bx_max = bp[2]; K.by_min = bp[3];
    K.T_sen = thresh_lt(d_sen);
    K.T_col = thresh_lt(K.two_size);
    const double d_near = d_sen + r_avoid / 2.0;                          // CPP:161
    K.T_near = thresh_lt(d_near);
    K.T_near_hi = (d_near * (1.0 + 1e-9)) * (d_near * (1.0 + 1e-9));
    K.U_occ = thresh_le(r_avoid / 2.0);                                   // CPP:185
    K.T_avoid = thresh_lt(r_avoid);                                       // CPP:482, 1166
    K.Tsen_f = std::nextafterf((float)(K.T_sen * (double)SLACK_REL + (double)SLACK_ABS), INFINITY);   // box test threshold
    // fp32 filter of the agent-pair loops: exact squared distance <= T  =>  fp32 squared distance <= T * (1 + 1e-4) + 1e-5
    // for |coordinates| < 16 (rounding of the positions to fp32: 2 * 16 * 2^-24 per difference, see k_step)
    auto pair_filter_threshold = [](double T) { return std::nextafterf((float)(T * 1.0001 + 1e-5), INFINITY); };
    K.Tcol_f = pair_filter_threshold(K.T_col);
    K.Tpair_f = pair_filter_threshold(std::max(K.T_sen, K.T_near_hi));
}

double in_shape_thresh(double l_cell) { return thresh_lt(std::sqrt(2.0) * l_cell / 2); }   // CPP:889

// Host mirror of the per-env match record (d_shape_id) that swarm_fast_path decides from.  It must never call an env matched that
// is not: the lookup kernel would index the table array with shape -1.  Every change goes through set(), which keeps the counts.
struct MatchMirror {
    enum State : unsigned char { UNMATCHED, DETECTED, EXACT };   // no library pose / pose detected (1e-9 accurate) / pose exact
    std::vector<State> env;
    long n_unposed = 0, n_inexact = 0;                           // envs UNMATCHED / not EXACT
    void init(int n) { env.assign(n, UNMATCHED); n_unposed = n_inexact = n; }
    void set(int e, State st) {
        n_unposed += (st == UNMATCHED) - (env[e] == UNMATCHED);
        n_inexact += (st != EXACT) - (env[e] != EXACT);
        env[e] = st;
    }
    void set_all(State st) { for (int e = 0; e < (int)env.size(); ++e) set(e, st); }
    static State of(int shape_id) { return shape_id < 0 ? UNMATCHED : (shape_id & POSE_EXACT) ? EXACT : DETECTED; }
};

}  // namespace

struct swarm_sim {
    swarm_config cfg;
    swarm_buffers buf;
    KParams K;
    int nt;                 // threads per CTA
    bool split;             // step = two launches (k_step PH 1 + PH 2)
    size_t smem1;           // dynamic shared memory of the first half
    size_t smem;            // dynamic shared memory of k_step PH 0
    size_t smem2;           // ... of the second-half kernel (PH 2)
    int pending;            // a_prior buffer holding the prior of the CURRENT state
    int last;               // a_prior buffer returned by the most recent step
    bool prior_dirty;       // state / grid changed behind the kernel's back
    bool observed;          // at least one observe/step ran (neighbor_index is meaningful)
    int64_t launches;
    double *d_stage; size_t stage_cap;     // set_grid staging (reference-layout grid)
    float *d_act; size_t act_cap;          // step_host action staging
    double *d_shape_grid; int *d_shape_ng; double *d_shape_thr; int n_shapes;   // swarm_set_shapes
    std::vector<double> shape_l_cell;
    // lookup scan: per-shape tables, per-env pose (library-owned device memory), host mirror of which envs are matched
    ShapeTab *d_tabs; std::vector<void *> tab_allocs; std::vector<ShapeTab> h_tabs;
    double4 *d_pose; int *d_shape_id;
    MatchMirror match;
    bool fast_ok;           // the shapes / sizes allow the lookup kernel at all
    bool all_tables;        // every library shape has a table (a reset cannot leave an env unmatched)
    bool xy_exact;          // every library shape has bit-identical x per lattice column and y per lattice row
    int rec_cap; size_t smem_fast;
    uint64_t lib_fp;        // fingerprint of the shape library (0: none), see library_fingerprint
};

// the k_step kernels launch_step runs for one step (dyn) or observe on a scan path (fast: see swarm_fast_path), and their dynamic
// shared memory; k1 = nullptr when the step is one launch.  The shared-memory limits are raised for exactly these kernels.
struct StepLaunch { step_fn_t k1, k2; size_t smem1, smem2; };
static StepLaunch step_launch(const swarm_sim *s, bool dyn, int fast) {
    const bool f32 = s->cfg.out_dtype == SWARM_F32, emit = s->cfg.emit_indices != 0;
    const size_t smem_scan = fast ? s->smem_fast : s->split ? s->smem2 : s->smem;
    // the second half runs no dynamics: observe and step share its DYN = false kernel
    if (s->split) return {step_kernel(f32, dyn, emit, 128, 1), step_kernel(f32, false, emit, 128, 2, fast), s->smem1, smem_scan};
    return {nullptr, step_kernel(f32, dyn, emit, (fast || s->nt > 128) ? 1024 : 128, 0, fast), 0, smem_scan};
}
static int raise_step_smem_limits(const swarm_sim *s, int fast) {
    for (int dyn = 0; dyn < 2; ++dyn) {
        const StepLaunch L = step_launch(s, dyn != 0, fast);
        if (L.k1) CU_TRY(raise_smem_limit((const void *)L.k1, L.smem1));
        CU_TRY(raise_smem_limit((const void *)L.k2, L.smem2));
    }
    return SWARM_OK;
}

extern "C" {

static int launch_step(swarm_sim *s, bool dyn, const void *act, int act_dtype, cudaStream_t st, const int32_t *env_list = nullptr,
                       int32_t count = 0);

/* shared with the other translation units of the library */
int swarm_set_last_error_(int code, const char *msg) { return fail(code, msg); }

int swarm_abi_version(void) { return 2; }
/* host-only helper exposed for tests: the squared-distance threshold equivalent to sqrt(s) < d (le=0) or <= d (le=1) */
double swarm_sqrt_threshold(double d, int le) { return le ? thresh_le(d) : thresh_lt(d); }
const char *swarm_last_error(void) { return g_last_error.c_str(); }
int32_t swarm_grid_pad(int32_t n_g_max) { return round32(n_g_max); }
int32_t swarm_obs_dim(const swarm_config *cfg) {
    if (cfg->variant == SWARM_VARIANT_FLOCKING) return 2 * 2 * (TOPO + (cfg->is_con_self_state ? 1 : 0));   // head rows only (VARIANTS.md 3)
    return 2 * 2 * (TOPO + 1 + (cfg->is_con_self_state ? 1 : 0)) + 2 * cfg->num_obs_grid_max;
}

int swarm_create(const swarm_config *cfg, const swarm_buffers *buf, swarm_sim **out) {
    if (!cfg || !buf || !out) return fail(SWARM_ERR_INVALID, "null argument");
    if (cfg->struct_size != (int32_t)sizeof(swarm_config) || buf->struct_size != (int32_t)sizeof(swarm_buffers))
        return fail(SWARM_ERR_INVALID, "struct_size mismatch (ABI)");
    if (cfg->num_envs <= 0 || cfg->n_a <= 0 || cfg->n_g_max <= 0) return fail(SWARM_ERR_INVALID, "sizes must be positive");
    if (cfg->topo_nei_max != TOPO) return fail(SWARM_ERR_UNSUPPORTED, "topo_nei_max must be 6");
    if (cfg->n_a > 1024) return fail(SWARM_ERR_UNSUPPORTED, "n_a > 1024 not supported by the fused kernel");
    if (cfg->num_obs_grid_max < 2 || cfg->num_occupied_grid_max < 2) return fail(SWARM_ERR_INVALID, "list caps must be >= 2");
    if (cfg->out_dtype != SWARM_F64 && cfg->out_dtype != SWARM_F32) return fail(SWARM_ERR_INVALID, "bad out_dtype");
    if (cfg->obs_layout != SWARM_OBS_REFERENCE && cfg->obs_layout != SWARM_OBS_AGENT_MAJOR) return fail(SWARM_ERR_INVALID, "bad obs_layout");
    if (cfg->variant != SWARM_VARIANT_ASSEMBLY && cfg->variant != SWARM_VARIANT_FLOCKING) return fail(SWARM_ERR_INVALID, "bad variant");
    if (cfg->variant == SWARM_VARIANT_FLOCKING && (cfg->n_a > 128 || cfg->emit_indices))
        return fail(SWARM_ERR_UNSUPPORTED, "the flocking variant supports n_a <= 128 and no index arrays");
    if (!buf->p || !buf->dp || !buf->grid || !buf->n_g || !buf->in_thresh || !buf->obs || !buf->reward ||
        !buf->a_prior[0] || !buf->a_prior[1] || !buf->neighbor_index || !buf->in_flags || !buf->word_box || !buf->frame ||
        !buf->nearest_cell)
        return fail(SWARM_ERR_INVALID, "required device buffer is NULL");
    if (cfg->emit_indices && (!buf->sensed_index || !buf->occupied_index))
        return fail(SWARM_ERR_INVALID, "emit_indices needs sensed_index / occupied_index buffers");

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(SWARM_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU fallback)");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(SWARM_ERR_INVALID, "device ordinal out of range");
    CU_TRY(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10) return fail(SWARM_ERR_NO_DEVICE, "device is not sm_100 (kernels are built for sm_100a only)");

    swarm_sim *s = new swarm_sim();
    s->cfg = *cfg; s->buf = *buf;
    memset(&s->K, 0, sizeof(KParams));
    fill_constants(s->K, cfg->n_a, cfg->n_g_max, cfg->num_obs_grid_max, cfg->num_occupied_grid_max,
                   cfg->is_con_self_state != 0, cfg->want_prior != 0, cfg->exact_occupancy != 0, cfg->is_periodic != 0, cfg->d_sen,
                   cfg->r_avoid, cfg->size_a, cfg->k_ball, cfg->k_wall, cfg->c_wall, cfg->dt, cfg->vel_max,
                   cfg->mass, cfg->boundary_pos);
    KParams &K = s->K;
    if (cfg->variant == SWARM_VARIANT_FLOCKING) K.obs_dim = swarm_obs_dim(cfg);
    K.E = cfg->num_envs;
    K.p = buf->p; K.dp = buf->dp; K.grid = reinterpret_cast<const double2 *>(buf->grid);
    K.n_g = buf->n_g; K.in_thresh = buf->in_thresh;
    K.wbox = reinterpret_cast<const float4 *>(buf->word_box); K.frame = buf->frame; K.brute_scan = cfg->brute_force_scan != 0; K.exact_reward = (cfg->debug_flags & 1) != 0; K.obs_am = cfg->obs_layout == SWARM_OBS_AGENT_MAJOR;
    K.obs = buf->obs; K.reward = buf->reward;
    K.nbr = buf->neighbor_index; K.in_flags = buf->in_flags; K.nearest = buf->nearest_cell;
    K.sensed = buf->sensed_index; K.occupied = buf->occupied_index;
    s->nt = round32(cfg->n_a);
    s->smem = step_smem_bytes(s->nt, K.n_words, cfg->emit_indices != 0, cfg->num_obs_grid_max);
    s->smem2 = step_smem_bytes(s->nt, K.n_words, cfg->emit_indices != 0, cfg->num_obs_grid_max, 2);
    s->smem1 = step_smem_bytes(s->nt, K.n_words, cfg->emit_indices != 0, cfg->num_obs_grid_max, 1);
    if (s->smem > (size_t)prop.sharedMemPerBlockOptin) {
        delete s;
        return fail(SWARM_ERR_UNSUPPORTED, "n_a x n_g_max needs more shared memory than one SM has");
    }
    s->split = (s->nt == 32) && !getenv("SWARM_FUSED_STEP");      // single-warp envs: two launches per step (see k_step, PH)
    if (const int rc = raise_step_smem_limits(s, 0)) { delete s; return rc; }
    s->pending = 0; s->last = 0; s->prior_dirty = true; s->observed = false; s->launches = 0;
    s->d_stage = nullptr; s->stage_cap = 0; s->d_act = nullptr; s->act_cap = 0;
    s->d_shape_grid = nullptr; s->d_shape_ng = nullptr; s->d_shape_thr = nullptr; s->n_shapes = 0;
    s->d_tabs = nullptr; s->d_pose = nullptr; s->d_shape_id = nullptr;
    s->match.init(cfg->num_envs);
    s->fast_ok = false; s->all_tables = false; s->xy_exact = false; s->rec_cap = 0; s->smem_fast = 0;
    s->lib_fp = 0;
    {
        cudaError_t e1 = cudaMalloc(&s->d_pose, sizeof(double4) * (size_t)cfg->num_envs);
        cudaError_t e2 = cudaMalloc(&s->d_shape_id, sizeof(int) * (size_t)cfg->num_envs);
        if (e1 == cudaSuccess && e2 == cudaSuccess) e1 = cudaMemset(s->d_shape_id, 0xFF, sizeof(int) * (size_t)cfg->num_envs);
        if (e1 != cudaSuccess || e2 != cudaSuccess) {
            if (s->d_pose) cudaFree(s->d_pose);
            if (s->d_shape_id) cudaFree(s->d_shape_id);
            delete s;
            return fail(SWARM_ERR_CUDA, "cudaMalloc of the pose arrays failed");
        }
    }
    s->K.pose = s->d_pose; s->K.shape_id = s->d_shape_id;
    *out = s;
    return SWARM_OK;
}

int swarm_destroy(swarm_sim *s) {
    if (!s) return SWARM_OK;
    cudaSetDevice(s->cfg.device);
    if (s->d_stage) cudaFree(s->d_stage);
    if (s->d_act) cudaFree(s->d_act);
    if (s->d_shape_grid) cudaFree(s->d_shape_grid);
    if (s->d_shape_ng) cudaFree(s->d_shape_ng);
    if (s->d_shape_thr) cudaFree(s->d_shape_thr);
    if (s->d_pose) cudaFree(s->d_pose);
    if (s->d_shape_id) cudaFree(s->d_shape_id);
    if (s->d_tabs) cudaFree(s->d_tabs);
    for (void *q : s->tab_allocs) cudaFree(q);
    delete s;
    return SWARM_OK;
}

/* reads back which of envs [env0, env0 + count) matched a library shape (d_shape_id, written by the kernels that build grids) into
 * the host mirror; synchronises the stream */
static int sync_match(swarm_sim *s, int32_t env0, int32_t count, cudaStream_t st) {
    std::vector<int> ids(count);
    CU_TRY(cudaMemcpyAsync(ids.data(), s->d_shape_id + env0, sizeof(int) * count, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    for (int k = 0; k < count; ++k) s->match.set(env0 + k, MatchMirror::of(ids[k]));
    return SWARM_OK;
}

int swarm_set_grid(swarm_sim *s, int32_t env0, int32_t count, const double *grid, int grid_on_device,
                   const int32_t *n_g, const double *l_cell, void *stream) {
    if (!s || !grid || !n_g || !l_cell) return fail(SWARM_ERR_INVALID, "null argument");
    if (env0 < 0 || count <= 0 || env0 + count > s->cfg.num_envs) return fail(SWARM_ERR_INVALID, "env range out of bounds");
    cudaStream_t st = (cudaStream_t)stream;
    CU_TRY(cudaSetDevice(s->cfg.device));
    const int ngm = s->cfg.n_g_max;
    std::vector<double> thr(count);
    for (int k = 0; k < count; ++k) {
        if (n_g[k] <= 0 || n_g[k] > ngm) return fail(SWARM_ERR_INVALID, "n_g out of range (0, n_g_max]");
        thr[k] = in_shape_thresh(l_cell[k]);
    }
    CU_TRY(cudaMemcpyAsync(s->buf.n_g + env0, n_g, sizeof(int32_t) * count, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(s->buf.in_thresh + env0, thr.data(), sizeof(double) * count, cudaMemcpyHostToDevice, st));
    const double *src = grid;
    if (!grid_on_device) {
        const size_t need = (size_t)count * 2 * ngm;
        if (const int rc = grow_staging(s->d_stage, s->stage_cap, need)) return rc;
        CU_TRY(cudaMemcpyAsync(s->d_stage, grid, need * sizeof(double), cudaMemcpyHostToDevice, st));
        src = s->d_stage;
    }
    PoseArgs A;
    A.n_shapes = s->fast_ok ? s->n_shapes : 0; A.n_g_cap = ngm;
    A.tabs = s->d_tabs; A.shape_grid = s->d_shape_grid; A.shape_n_g = s->d_shape_ng;
    A.pose = s->d_pose + env0; A.shape_id = s->d_shape_id + env0;
    k_pack_grid<<<count, 128, 0, st>>>(src, (long)2 * ngm, s->buf.n_g + env0, s->K.n_g_pad,
                                       reinterpret_cast<double2 *>(s->buf.grid) + (size_t)env0 * s->K.n_g_pad,
                                       reinterpret_cast<float4 *>(s->buf.word_box) + (size_t)env0 * s->K.n_words,
                                       s->buf.frame + (size_t)env0 * 2, A);
    CU_TRY(cudaGetLastError());
    s->launches++;
    // which of these envs matched a library shape (lookup scan) — the host mirror decides which kernel a step launches.
    // (its stream sync also keeps the thr/n_g host vectors alive until the async copies are done)
    if (const int rc = sync_match(s, env0, count, st)) return rc;
    s->prior_dirty = true;
    return SWARM_OK;
}

static int install_shapes(swarm_sim *s, int32_t n_shapes, const double *grids, const int32_t *n_g, const double *l_cell) {
    if (!s || !grids || !n_g || !l_cell || n_shapes <= 0) return fail(SWARM_ERR_INVALID, "bad argument");
    CU_TRY(cudaSetDevice(s->cfg.device));
    const int ngm = s->cfg.n_g_max;
    std::vector<double> thr(n_shapes);
    for (int k = 0; k < n_shapes; ++k) {
        if (n_g[k] <= 0 || n_g[k] > ngm) return fail(SWARM_ERR_INVALID, "shape n_g out of range (0, n_g_max]");
        thr[k] = in_shape_thresh(l_cell[k]);
    }
    if (s->d_shape_grid) { cudaFree(s->d_shape_grid); cudaFree(s->d_shape_ng); cudaFree(s->d_shape_thr); }
    s->d_shape_grid = nullptr; s->d_shape_ng = nullptr; s->d_shape_thr = nullptr; s->n_shapes = 0;
    CU_TRY(cudaMalloc(&s->d_shape_grid, sizeof(double) * (size_t)n_shapes * 2 * ngm));
    CU_TRY(cudaMalloc(&s->d_shape_ng, sizeof(int) * n_shapes));
    CU_TRY(cudaMalloc(&s->d_shape_thr, sizeof(double) * n_shapes));
    CU_TRY(cudaMemcpy(s->d_shape_grid, grids, sizeof(double) * (size_t)n_shapes * 2 * ngm, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(s->d_shape_ng, n_g, sizeof(int) * n_shapes, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(s->d_shape_thr, thr.data(), sizeof(double) * n_shapes, cudaMemcpyHostToDevice));
    s->n_shapes = n_shapes;
    s->shape_l_cell.assign(l_cell, l_cell + n_shapes);

    // ---- lookup-scan tables (see ShapeTab / k_build_bins).  Any earlier pose refers to the old library: forget it.
    for (void *q : s->tab_allocs) cudaFree(q);
    s->tab_allocs.clear();
    if (s->d_tabs) { cudaFree(s->d_tabs); s->d_tabs = nullptr; }
    CU_TRY(cudaMemset(s->d_shape_id, 0xFF, sizeof(int) * (size_t)s->cfg.num_envs));
    s->match.set_all(MatchMirror::UNMATCHED);
    s->fast_ok = false; s->all_tables = false; s->xy_exact = true;
    s->h_tabs.assign(n_shapes, ShapeTab{});
    // the lookup kernel serves single-warp envs with <= 1024 cells; rows per agent <= 32 and cells per row record <= 31
    double l_min = l_cell[0];
    for (int k = 1; k < n_shapes; ++k) l_min = std::min(l_min, l_cell[k]);
    const double rr = s->cfg.d_sen / l_min;
    // (the lookup scan finds covered cells among an agent's sensing candidates: the covering radius must be the smaller one)
    const bool eligible = ((s->split && s->nt == 32) || (!s->split && s->nt > 32)) && s->K.n_words <= 32 && ngm <= 1023 && rr <= 14.9 && !s->cfg.brute_force_scan &&
                          0.5 * s->cfg.r_avoid + 1e-6 < s->cfg.d_sen &&
                          !getenv("SWARM_NO_LOOKUP_SCAN");
    if (!eligible) return SWARM_OK;
    const double half_extent = std::max(s->K.half_w, s->K.half_h);
    // origin-frame positions the table must cover: |p| up to the walls (+ slack: they are soft), |offset| up to half - 1 (ENV:184-185)
    const double Q = 1.4142135623730951 * ((half_extent + 0.25) + std::max(half_extent - 1.0, 0.0)) + 0.1;
    int n_tables = 0, lat_n = 8;
    struct HostLattice { std::vector<double> colx, rowy; std::vector<unsigned long long> rowmask; std::vector<unsigned short> rowstart; };
    std::vector<HostLattice> lat(n_shapes);
    for (int k = 0; k < n_shapes; ++k) {
        const double *gx = grids + (size_t)k * 2 * ngm, *gy = gx + n_g[k];
        const int n = n_g[k];
        const double L = l_cell[k];
        ShapeTab &T = s->h_tabs[k];
        double ox_min = gx[0], oy_min = gy[0];
        for (int c = 0; c < n; ++c) { ox_min = std::min(ox_min, gx[c]); oy_min = std::min(oy_min, gy[c]); }
        // lattice recovery: every cell at (ox_min + ix L, oy_min + iy L), numbered row by row
        bool ok = L > 0 && n >= 2;
        std::vector<unsigned long long> rowmask;
        std::vector<unsigned short> rowstart;
        int ncols = 0, far_cell = 0; long prev_key = -1; double far_d2 = -1.0;
        for (int c = 0; c < n && ok; ++c) {
            const long ix = std::lround((gx[c] - ox_min) / L), iy = std::lround((gy[c] - oy_min) / L);
            ok = ix >= 0 && ix < 64 && iy >= 0 && iy < 64 && std::fabs(gx[c] - (ox_min + ix * L)) <= 1e-9 &&
                 std::fabs(gy[c] - (oy_min + iy * L)) <= 1e-9 && iy * 64 + ix > prev_key;
            if (!ok) break;
            prev_key = iy * 64 + ix;
            if ((long)rowmask.size() <= iy) { rowmask.resize(iy + 1, 0ull); rowstart.resize(iy + 1, (unsigned short)c); }
            if (rowmask[iy] == 0ull) rowstart[iy] = (unsigned short)c;
            rowmask[iy] |= 1ull << ix;
            ncols = std::max(ncols, (int)ix + 1);
            const double d2 = (gx[c] - gx[0]) * (gx[c] - gx[0]) + (gy[c] - gy[0]) * (gy[c] - gy[0]);
            if (d2 > far_d2) { far_d2 = d2; far_cell = c; }
        }
        if (!ok || far_cell == 0) continue;                          // not a lattice shape: its envs use the general scan
        for (size_t r = 0; r < rowmask.size(); ++r) if (rowmask[r] == 0ull) rowstart[r] = (r ? rowstart[r - 1] : 0);
        const int nrows = (int)rowmask.size();
        rowmask.resize(64, 0ull); rowstart.resize(64, (unsigned short)n);
        // exact column / row coordinates: every cell of column ix has the same x bits, every cell of row iy the same y bits
        // (true for grids generated like assembly_cfg.py:44-99); otherwise the exact-pose kernel variant is not used
        std::vector<double> colx(64, 0.0), rowy(64, 0.0);
        std::vector<char> cset(64, 0), rset(64, 0);
        for (int c = 0; c < n; ++c) {
            const long ix = std::lround((gx[c] - ox_min) / L), iy = std::lround((gy[c] - oy_min) / L);
            if (!cset[ix]) { cset[ix] = 1; colx[ix] = gx[c]; }
            if (!rset[iy]) { rset[iy] = 1; rowy[iy] = gy[c]; }
            if (colx[ix] != gx[c] || rowy[iy] != gy[c]) s->xy_exact = false;
        }
        const double h = 0.5 * L;
        const int nb = (int)std::ceil(2.0 * Q / h);
        if ((size_t)nb * nb > (size_t)4 << 20) continue;             // table would be unreasonably large
        unsigned short *d_spill = nullptr; uint2 *d_bins = nullptr;
        double2 *d_cells = nullptr;
        std::vector<double2> cells(n);
        for (int c = 0; c < n; ++c) cells[c] = make_double2(gx[c], gy[c]);
        CU_TRY(cudaMalloc(&d_cells, sizeof(double2) * n)); s->tab_allocs.push_back(d_cells);
        CU_TRY(cudaMemcpy(d_cells, cells.data(), sizeof(double2) * n, cudaMemcpyHostToDevice));
        unsigned *d_cursor = nullptr;
        const unsigned spill_cap = (unsigned)nb * nb * 2u;
        CU_TRY(cudaMalloc(&d_bins, sizeof(uint2) * (size_t)nb * nb)); s->tab_allocs.push_back(d_bins);
        CU_TRY(cudaMalloc(&d_spill, sizeof(unsigned short) * (size_t)spill_cap)); s->tab_allocs.push_back(d_spill);
        CU_TRY(cudaMalloc(&d_cursor, sizeof(unsigned))); s->tab_allocs.push_back(d_cursor);
        CU_TRY(cudaMemset(d_cursor, 0, sizeof(unsigned)));
        k_build_bins<<<(nb * nb + 127) / 128, 128>>>(s->d_shape_grid + (size_t)k * 2 * ngm, n, -Q, h, nb, d_bins, d_spill, d_cursor, spill_cap);
        CU_TRY(cudaGetLastError());
        s->launches++;
        T.ox_min = ox_min; T.oy_min = oy_min; T.inv_l = 1.0 / L; T.q0 = -Q; T.inv_h = 1.0 / h;
        T.ncols = ncols; T.nrows = nrows; T.nb = nb; T.far_cell = far_cell;
        lat[k].colx = colx; lat[k].rowy = rowy; lat[k].rowmask = rowmask; lat[k].rowstart = rowstart;
        lat_n = std::max(lat_n, (std::max(ncols, nrows) + 7) & ~7);
        T.bins = d_bins; T.spill = d_spill; T.cells = d_cells;
        ++n_tables;
    }
    CU_TRY(cudaDeviceSynchronize());
    s->all_tables = n_tables == n_shapes;
    if (n_tables == 0) return SWARM_OK;
    // lattice blobs, all with lat_n entries per table (see ShapeTab::lattice)
    for (int k = 0; k < n_shapes; ++k) {
        if (!s->h_tabs[k].nb) continue;
        const int words = 3 * lat_n + lat_n / 4;
        std::vector<unsigned long long> blob(words, 0ull);
        memcpy(blob.data(), lat[k].colx.data(), 8 * lat_n); memcpy(blob.data() + lat_n, lat[k].rowy.data(), 8 * lat_n);
        memcpy(blob.data() + 2 * lat_n, lat[k].rowmask.data(), 8 * lat_n); memcpy(blob.data() + 3 * lat_n, lat[k].rowstart.data(), 2 * lat_n);
        unsigned long long *d_blob = nullptr;
        CU_TRY(cudaMalloc(&d_blob, sizeof(unsigned long long) * words)); s->tab_allocs.push_back(d_blob);
        CU_TRY(cudaMemcpy(d_blob, blob.data(), sizeof(unsigned long long) * words, cudaMemcpyHostToDevice));
        s->h_tabs[k].lattice = d_blob;
    }
    s->K.lat_n = lat_n;
    CU_TRY(cudaMalloc(&s->d_tabs, sizeof(ShapeTab) * n_shapes));
    CU_TRY(cudaMemcpy(s->d_tabs, s->h_tabs.data(), sizeof(ShapeTab) * n_shapes, cudaMemcpyHostToDevice));
    s->K.shapes = s->d_tabs;
    s->K.n_tab_inline = std::min(n_shapes, (int)TAB_INLINE);
    for (int k = 0; k < s->K.n_tab_inline; ++k) s->K.tab_inline[k] = s->h_tabs[k];
    const int rows_per_agent = (2.0 * (rr + 2e-3) + 2.0 <= 16.0) ? 16 : 32;
    s->rec_cap = 32 * rows_per_agent;                              // per warp
    s->K.rec_cap = s->rec_cap;
    s->smem_fast = step_smem_bytes(s->nt, s->K.n_words, s->cfg.emit_indices != 0, s->cfg.num_obs_grid_max, s->split ? 2 : 0, s->rec_cap, lat_n);
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, s->cfg.device));
    if (s->smem_fast > (size_t)prop.sharedMemPerBlockOptin) return SWARM_OK;      // does not fit (e.g. 1024 agents with index arrays): general scan
    for (int fast = 1; fast <= 2; ++fast)
        if (const int rc = raise_step_smem_limits(s, fast)) return rc;
    s->fast_ok = true;
    return SWARM_OK;
}

/* What a shape id means on this handle: a hash of the library (shape count, cells, cell sizes) and of which shapes the lookup
 * scan serves.  A state saved under one fingerprint keeps its match record only when loaded under the same one (DESIGN.md §11). */
static uint64_t library_fingerprint(const swarm_sim *s, const double *grids, const int32_t *n_g, const double *l_cell) {
    uint64_t h = 1469598103934665603ull;                                      // FNV-1a
    auto mix = [&h](const void *p, size_t n) {
        for (size_t i = 0; i < n; ++i) { h ^= static_cast<const unsigned char *>(p)[i]; h *= 1099511628211ull; }
    };
    mix(&s->n_shapes, sizeof(int));
    for (int k = 0; k < s->n_shapes; ++k) {
        mix(&n_g[k], sizeof(int32_t)); mix(&l_cell[k], sizeof(double));
        mix(grids + (size_t)k * 2 * s->cfg.n_g_max, sizeof(double) * 2 * (size_t)n_g[k]);
        const unsigned char tab = s->h_tabs[k].nb != 0;
        mix(&tab, 1);
    }
    const unsigned char ok = s->fast_ok;
    mix(&ok, 1);
    h &= ~(1ull << 63);
    return h ? h : 1;
}

int swarm_set_shapes(swarm_sim *s, int32_t n_shapes, const double *grids, const int32_t *n_g, const double *l_cell) {
    const int rc = install_shapes(s, n_shapes, grids, n_g, l_cell);
    if (rc == SWARM_OK) s->lib_fp = library_fingerprint(s, grids, n_g, l_cell);
    else if (rc != SWARM_ERR_INVALID) {        // failed half way: a library no saved state can claim
        static std::atomic<uint64_t> failed{0};
        s->lib_fp = (1ull << 63) | ++failed;
    }
    return rc;
}

/* Target shapes for envs [env0, env0 + count) given as (library shape, pose): grid_center = R * origin + off computed on the
 * device with the reference's roundings (ENV:175-187).  shape_ids [count] and pose [count][4] = (cos, sin, off_x, off_y) are
 * HOST arrays.  Equivalent to swarm_set_grid with that grid, but the pose is then known exactly (see swarm_fast_path). */
int swarm_set_grid_pose(swarm_sim *s, int32_t env0, int32_t count, const int32_t *shape_ids, const double *pose, void *stream) {
    if (!s || !shape_ids || !pose) return fail(SWARM_ERR_INVALID, "null argument");
    if (env0 < 0 || count <= 0 || env0 + count > s->cfg.num_envs) return fail(SWARM_ERR_INVALID, "env range out of bounds");
    if (s->n_shapes <= 0) return fail(SWARM_ERR_INVALID, "swarm_set_grid_pose before swarm_set_shapes");
    for (int k = 0; k < count; ++k)
        if (shape_ids[k] < 0 || shape_ids[k] >= s->n_shapes) return fail(SWARM_ERR_INVALID, "shape id out of range");
    cudaStream_t st = (cudaStream_t)stream;
    CU_TRY(cudaSetDevice(s->cfg.device));
    const size_t need = (size_t)count * 5;                       // staging: ids (as doubles' worth of space) + poses
    if (const int rc = grow_staging(s->d_stage, s->stage_cap, need)) return rc;
    double4 *d_pose_in = reinterpret_cast<double4 *>(s->d_stage);
    int *d_ids = reinterpret_cast<int *>(s->d_stage + (size_t)count * 4);
    CU_TRY(cudaMemcpyAsync(d_pose_in, pose, sizeof(double) * 4 * count, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(d_ids, shape_ids, sizeof(int) * count, cudaMemcpyHostToDevice, st));
    k_grid_from_pose<<<count, 128, 0, st>>>(s->K.n_g_pad, s->cfg.n_g_max, s->d_shape_grid, s->d_shape_ng, s->d_shape_thr,
                                            s->fast_ok ? s->d_tabs : nullptr, d_ids, d_pose_in,
                                            reinterpret_cast<double2 *>(s->buf.grid) + (size_t)env0 * s->K.n_g_pad, s->buf.n_g + env0,
                                            s->buf.in_thresh + env0, reinterpret_cast<float4 *>(s->buf.word_box) + (size_t)env0 * s->K.n_words,
                                            s->buf.frame + (size_t)env0 * 2, s->d_pose + env0, s->d_shape_id + env0);
    CU_TRY(cudaGetLastError());
    s->launches++;
    if (const int rc = sync_match(s, env0, count, st)) return rc;   // (its stream sync also lets the caller free the host arrays)
    s->prior_dirty = true;
    return SWARM_OK;
}

/* which second-half kernel the next swarm_step / swarm_observe runs: 0 = general culled scan, 1 = lookup scan on the stored
 * cells (every env's grid matched a library shape), 2 = lookup scan with cells recomputed from the library (every pose exact) */
int swarm_fast_path(const swarm_sim *s) {
    if (!(s && s->fast_ok && s->match.n_unposed == 0)) return 0;
    return (s->match.n_inexact == 0 && s->xy_exact) ? 2 : 1;
}

/* the k_reset arguments of swarm_reset / swarm_reset_envs: every env (env_mask and env_list NULL), the masked envs or the listed ones */
static ResetParams reset_params(const swarm_sim *s, uint64_t seed, uint64_t episode, uint64_t env_offset, const uint8_t *env_mask,
                                const int32_t *env_list, double *info_dev) {
    ResetParams R;
    R.n_a = s->cfg.n_a; R.n_g_pad = s->K.n_g_pad; R.n_g_cap = s->cfg.n_g_max; R.n_shapes = s->n_shapes;
    R.half_w = s->K.half_w; R.half_h = s->K.half_h;
    R.shape_grid = s->d_shape_grid; R.shape_n_g = s->d_shape_ng; R.shape_thresh = s->d_shape_thr;
    R.p = s->buf.p; R.dp = s->buf.dp; R.grid = reinterpret_cast<double2 *>(s->buf.grid); R.n_g = s->buf.n_g;
    R.in_thresh = s->buf.in_thresh; R.wbox = reinterpret_cast<float4 *>(s->buf.word_box); R.frame = s->buf.frame;
    R.nearest = s->buf.nearest_cell; R.info = info_dev; R.mask = env_mask; R.env_list = env_list;
    R.seed = seed; R.episode = episode; R.env_offset = env_offset;
    R.pose = s->fast_ok ? s->d_pose : nullptr; R.shape_id = s->fast_ok ? s->d_shape_id : nullptr; R.tabs = s->d_tabs;
    return R;
}

int swarm_reset(swarm_sim *s, uint64_t seed, uint64_t episode, uint64_t env_offset, const uint8_t *env_mask,
                double *info_dev, void *stream) {
    if (!s) return fail(SWARM_ERR_INVALID, "null handle");
    if (s->n_shapes <= 0) return fail(SWARM_ERR_INVALID, "swarm_reset before swarm_set_shapes");
    CU_TRY(cudaSetDevice(s->cfg.device));
    k_reset<<<s->cfg.num_envs, 128, 0, (cudaStream_t)stream>>>(reset_params(s, seed, episode, env_offset, env_mask, nullptr, info_dev));
    CU_TRY(cudaGetLastError());
    s->launches++;
    s->prior_dirty = true;
    if (s->fast_ok) {
        if (!s->all_tables) {
            // an env that drew a shape without a table is unmatched now: the observe below must not run the lookup scan on it
            if (const int rc = sync_match(s, 0, s->cfg.num_envs, (cudaStream_t)stream)) return rc;
        } else if (!env_mask) {
            // every env now has an exact library pose.  (A masked reset keeps the mirror: it only makes unmatched envs matched)
            s->match.set_all(MatchMirror::EXACT);
        }
    }
    return swarm_observe(s, stream);     // ENV:221; a masked reset re-observes every env (idempotent for the untouched ones)
}

/* swarm_reset for a LIST of envs (device int32 array, no duplicates): only those envs are re-randomised and re-observed,
 * one CTA each — the auto-reset of a vector env whose episodes end at different steps. */
int swarm_reset_envs(swarm_sim *s, uint64_t seed, uint64_t episode, uint64_t env_offset, const int32_t *env_list_dev, int32_t count,
                     double *info_dev, void *stream) {
    if (!s || !env_list_dev) return fail(SWARM_ERR_INVALID, "null argument");
    if (count <= 0 || count > s->cfg.num_envs) return fail(SWARM_ERR_INVALID, "count out of range");
    if (s->n_shapes <= 0) return fail(SWARM_ERR_INVALID, "swarm_reset_envs before swarm_set_shapes");
    if (!s->observed) return fail(SWARM_ERR_INVALID, "swarm_reset_envs needs a full reset / observe first");
    CU_TRY(cudaSetDevice(s->cfg.device));
    k_reset<<<count, 128, 0, (cudaStream_t)stream>>>(reset_params(s, seed, episode, env_offset, nullptr, env_list_dev, info_dev));
    CU_TRY(cudaGetLastError());
    s->launches++;
    // When every library shape has a table, the host keeps its matched-env count without a sync: matched envs stay matched;
    // unmatched ones in the list become matched on the device, which the host does not track, so the general kernel stays in
    // use until a full reset / set_grid.  Otherwise a listed env may have drawn a shape without a table and become unmatched:
    // the mirror is read back before the observe below picks its kernel.
    if (s->fast_ok && !s->all_tables)
        if (const int rc = sync_match(s, 0, s->cfg.num_envs, (cudaStream_t)stream)) return rc;
    // observation + prior of the new state for the listed envs only; the others keep theirs (the a_prior buffer written is the
    // one holding the prior of the CURRENT state, which the next step returns)
    return launch_step(s, false, nullptr, SWARM_F32, (cudaStream_t)stream, env_list_dev, count);
}

/* measurement aid: dense FMA throughput of this device (TFLOP/s), fp32 and fp64 — the roofline denominator of the O(n_a^2)
 * configuration (SURVEY.md 8(d)); best of 3 timed launches each */
int swarm_measure_fma_peak(int32_t device, double *fp32_tflops, double *fp64_tflops) {
    if (!fp32_tflops || !fp64_tflops) return fail(SWARM_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    void *sink = nullptr;
    CU_TRY(cudaMalloc(&sink, 64));
    cudaEvent_t a, b;
    CU_TRY(cudaEventCreate(&a)); CU_TRY(cudaEventCreate(&b));
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    double best[2] = {0.0, 0.0};
    for (int which = 0; which < 2; ++which) {
        const int iters = which ? 1 << 14 : 1 << 17;
        for (int rep = 0; rep < 4; ++rep) {
            CU_TRY(cudaEventRecord(a));
            if (which) k_fma_peak<double><<<blocks, threads>>>(iters, (double *)sink);
            else k_fma_peak<float><<<blocks, threads>>>(iters, (float *)sink);
            CU_TRY(cudaEventRecord(b));
            CU_TRY(cudaEventSynchronize(b));
            float ms = 0.f;
            CU_TRY(cudaEventElapsedTime(&ms, a, b));
            const double tf = (double)blocks * threads * (double)iters * 16.0 / (ms * 1e-3) / 1e12;
            if (rep > 0 && tf > best[which]) best[which] = tf;
        }
    }
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(sink);
    *fp32_tflops = best[0]; *fp64_tflops = best[1];
    return SWARM_OK;
}

/* self-test: the shared-reciprocal division of the prior (div_shared) against a / b on n pseudo-random operand pairs */
int swarm_selftest_division(int32_t device, uint64_t n, uint64_t seed, int32_t kind, uint64_t *mismatches) {
    if (!mismatches || kind < 0 || kind > 2) return fail(SWARM_ERR_INVALID, "bad argument");
    CU_TRY(cudaSetDevice(device));
    unsigned long long *d = nullptr;
    CU_TRY(cudaMalloc(&d, sizeof(unsigned long long)));
    CU_TRY(cudaMemset(d, 0, sizeof(unsigned long long)));
    k_selftest_division<<<1184, 256>>>((unsigned long long)n, (unsigned long long)seed, kind, d);
    unsigned long long h = 0;
    cudaError_t e = cudaMemcpy(&h, d, sizeof(h), cudaMemcpyDeviceToHost);
    cudaFree(d);
    CU_TRY(e);
    *mismatches = h;
    return SWARM_OK;
}

int swarm_metrics(swarm_sim *s, double *out_dev, void *stream) {
    if (!s || !out_dev) return fail(SWARM_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(s->cfg.device));
    const int n_a = s->cfg.n_a;
    const size_t smem = (size_t)3 * n_a * sizeof(double) + (size_t)(n_a + 2) * sizeof(int);
    k_metrics<<<s->cfg.num_envs, 128, smem, (cudaStream_t)stream>>>(n_a, s->K.p, s->K.grid, s->K.n_g_pad, s->K.n_g,
                                                                    thresh_lt(s->cfg.r_avoid / 2), out_dev);
    CU_TRY(cudaGetLastError());
    s->launches++;
    return SWARM_OK;
}

int swarm_render_palette(uint8_t *rgb) {
    static const uint8_t pal[RC_COUNT * 3] = {SWARM_RGB_ARENA, SWARM_RGB_OUTSIDE, SWARM_RGB_CELL, SWARM_RGB_TRAIL,
                                              SWARM_RGB_AGENT_IN, SWARM_RGB_AGENT_OUT};
    if (rgb) memcpy(rgb, pal, sizeof(pal));
    return RC_COUNT;
}

int swarm_render(swarm_sim *s, const swarm_render_args *a, void *stream) {
    if (!s || !a) return fail(SWARM_ERR_INVALID, "null argument");
    if (a->struct_size != (int32_t)sizeof(swarm_render_args)) return fail(SWARM_ERR_INVALID, "struct_size mismatch (ABI)");
    if (a->width < 1 || a->width > 8192 || a->height < 1 || a->height > 8192)
        return fail(SWARM_ERR_INVALID, "width and height must be in [1, 8192]");
    if (a->flags & ~(SWARM_RENDER_CELLS | SWARM_RENDER_AGENTS | SWARM_RENDER_TRAILS)) return fail(SWARM_ERR_INVALID, "unknown flags");
    if (a->count < 1 || !a->env_ids) return fail(SWARM_ERR_INVALID, "count must be >= 1 with a non-NULL env_ids");
    for (int f = 0; f < a->count; ++f)
        if (a->env_ids[f] < 0 || a->env_ids[f] >= s->cfg.num_envs) return fail(SWARM_ERR_INVALID, "env id out of range");
    const double *bp = s->cfg.boundary_pos;
    const bool arena = a->view[0] == 0 && a->view[1] == 0 && a->view[2] == 0 && a->view[3] == 0;
    const double *v = arena ? bp : a->view;
    const double sx = (v[2] - v[0]) / a->width, sy = (v[1] - v[3]) / a->height;
    for (int k = 0; k < 4; ++k)
        if (!std::isfinite(v[k])) return fail(SWARM_ERR_INVALID, "view must be finite");
    if (!(v[0] < v[2] && v[3] < v[1]) || !std::isfinite(sx) || !std::isfinite(sy) || !(sx > 0) || !(sy > 0))
        return fail(SWARM_ERR_INVALID, "view needs xmin < xmax and ymin < ymax");
    if (a->trail_len < 0 || a->trail_len > a->trail_cap || a->trail_cap > 1024)
        return fail(SWARM_ERR_INVALID, "trail: 0 <= trail_len <= trail_cap <= 1024");
    if (a->trail_len > 0 && (!a->trail || a->trail_head < 0 || a->trail_head >= a->trail_cap))
        return fail(SWARM_ERR_INVALID, "trail: a non-NULL ring and 0 <= trail_head < trail_cap");
    if (!a->frames) return fail(SWARM_ERR_INVALID, "frames is NULL");
    CU_TRY(cudaSetDevice(s->cfg.device));

    RenderParams P{};
    const double size_a = s->cfg.size_a;
    P.W = a->width; P.H = a->height; P.flags = a->flags; P.n_a = s->cfg.n_a; P.n_g_pad = s->K.n_g_pad; P.count = a->count;
    P.cells_ok = s->cfg.variant == SWARM_VARIANT_ASSEMBLY;
    P.trail_cap = a->trail_cap; P.trail_len = a->trail_len; P.trail_head = a->trail_head;
    P.x0 = v[0]; P.y1 = v[1]; P.sx = sx; P.sy = sy;
    // cull margin: one pixel, plus slack for the roundings of the (inexact) box tests
    const double slack = 1e-12 * (std::fabs(v[0]) + std::fabs(v[1]) + std::fabs(v[2]) + std::fabs(v[3]) + 1.0);
    P.mx = sx + slack; P.my = sy + slack;
    P.ax0 = bp[0]; P.ay1 = bp[1]; P.ax1 = bp[2]; P.ay0 = bp[3];
    P.rr_agent = size_a * size_a; P.r_agent = size_a;
    P.w = size_a * 0.25; P.ww = P.w * P.w;
    P.half_w = s->K.half_w; P.half_h = s->K.half_h;
    P.p = s->buf.p; P.in_flags = s->buf.in_flags; P.grid = reinterpret_cast<const double2 *>(s->buf.grid);
    P.n_g = s->buf.n_g; P.in_thresh = s->buf.in_thresh;
    P.trail = a->trail; P.frames = a->frames;
    swarm_render_palette(&P.palette[0][0]);
    const dim3 tiles((a->width + RENDER_TILE - 1) / RENDER_TILE, (a->height + RENDER_TILE - 1) / RENDER_TILE);
    for (int f0 = 0; f0 < a->count; f0 += RENDER_IDS_PER_LAUNCH) {
        const int n = std::min(a->count - f0, RENDER_IDS_PER_LAUNCH);
        P.f0 = f0;
        memcpy(P.env, a->env_ids + f0, sizeof(int32_t) * n);
        k_render<<<dim3(tiles.x, tiles.y, n), RENDER_THREADS, 0, (cudaStream_t)stream>>>(P);
        CU_TRY(cudaGetLastError());
        s->launches++;
    }
    return SWARM_OK;
}

int swarm_strategy_actions(swarm_sim *s, int kind, double *act_dev, void *stream) {
    if (!s || !act_dev) return fail(SWARM_ERR_INVALID, "null argument");
    if (kind != SWARM_STRATEGY_RULE && kind != SWARM_STRATEGY_LLM) return fail(SWARM_ERR_INVALID, "kind must be SWARM_STRATEGY_RULE or SWARM_STRATEGY_LLM");
    if (kind == SWARM_STRATEGY_LLM && !s->observed) return fail(SWARM_ERR_INVALID, "the 'llm' strategy needs the neighbour list of an observation");
    if (s->cfg.is_periodic) return fail(SWARM_ERR_UNSUPPORTED, "strategies are implemented for is_boundary=True (the reference's Python twins never wrap)");
    CU_TRY(cudaSetDevice(s->cfg.device));
    const int n_a = s->cfg.n_a, th = n_a < 256 ? round32(n_a) : 256;
    if (kind == SWARM_STRATEGY_RULE)
        k_strategy<1><<<s->cfg.num_envs, th, 0, (cudaStream_t)stream>>>(n_a, TOPO, s->K.p, s->K.dp, s->K.grid, s->K.n_g_pad, s->K.n_g, s->K.in_thresh,
                                                                      s->K.nbr, s->K.d_sen, s->K.r_avoid, s->K.n_obs_max, act_dev);
    else
        k_strategy<2><<<s->cfg.num_envs, th, 0, (cudaStream_t)stream>>>(n_a, TOPO, s->K.p, s->K.dp, s->K.grid, s->K.n_g_pad, s->K.n_g, s->K.in_thresh,
                                                                      s->K.nbr, s->K.d_sen, s->K.r_avoid, s->K.n_obs_max, act_dev);
    CU_TRY(cudaGetLastError());
    s->launches++;
    return SWARM_OK;
}

int swarm_set_obs_buffer(swarm_sim *s, void *obs_dev) {
    if (!s || !obs_dev) return fail(SWARM_ERR_INVALID, "null argument");
    s->buf.obs = obs_dev; s->K.obs = obs_dev;
    return SWARM_OK;
}

int swarm_mark_state_dirty(swarm_sim *s) {
    if (!s) return fail(SWARM_ERR_INVALID, "null handle");
    s->prior_dirty = true;
    return SWARM_OK;
}

int swarm_restore_observation(swarm_sim *s) {
    if (!s) return fail(SWARM_ERR_INVALID, "null handle");
    s->observed = true;
    s->prior_dirty = true;       // the prior of the restored state is computed by k_prior at the next step (ENV:613-624)
    return SWARM_OK;
}

int swarm_is_observed(const swarm_sim *s) { return (s && s->observed) ? 1 : 0; }

}  // extern "C"

// ---- state store (DESIGN.md §11).  The segments of a slot, in slot order: one env row of each of these arrays.
enum StateSegId { SEG_P, SEG_DP, SEG_GRID, SEG_WBOX, SEG_FRAME, SEG_NG, SEG_THRESH, SEG_POSE, SEG_SHAPE, SEG_NEAREST, SEG_NBR,
                  SEG_FLAGS, SEG_OBS, SEG_REWARD, SEG_PRIOR_CUR, SEG_PRIOR_LAST, SEG_SENSED, SEG_OCC, SEG_COUNT };
static_assert(SEG_COUNT <= STATE_MAX_SEGS, "StateCopyParams::seg too small");

struct swarm_state_store {
    swarm_config cfg;                         // the configuration it serves (num_envs is not part of it)
    int64_t capacity;
    long long row[SEG_COUNT], off[SEG_COUNT]; // bytes per env row (0: not stored) and offset in the slot
    long long slot_bytes;
    int n_sm;
    unsigned char *d_slots;
    struct Slot {
        bool filled = false;
        bool prior_valid = false;             // the source's a_prior[pending] was the prior of its state (!prior_dirty)
        MatchMirror::State match = MatchMirror::UNMATCHED;   // the source env's mirror entry: never more than the device record
        uint64_t lib_fp = 0;                  // the source's library_fingerprint
    };
    std::vector<Slot> slot;
};

static bool same_config(const swarm_config &a, const swarm_config &b) {
    swarm_config x = a, y = b;
    x.num_envs = y.num_envs = 0;
    return memcmp(&x, &y, sizeof(swarm_config)) == 0;
}

// env row e of segment g of the handle starts at state_seg_base(s, g) + e * row[g]
static unsigned char *state_seg_base(const swarm_sim *s, int g) {
    const swarm_buffers &b = s->buf;
    void *const base[SEG_COUNT] = {b.p, b.dp, b.grid, b.word_box, b.frame, b.n_g, b.in_thresh, s->d_pose, s->d_shape_id,
                                   b.nearest_cell, b.neighbor_index, b.in_flags, b.obs, b.reward, b.a_prior[s->pending],
                                   b.a_prior[s->last], b.sensed_index, b.occupied_index};
    return static_cast<unsigned char *>(base[g]);
}

// checks shared by save and load: handle, store, lists; `distinct` names the list that must not repeat an id
static int state_check(const swarm_sim *s, const swarm_state_store *st, const int32_t *env_ids, const int32_t *slots, int32_t count,
                       bool envs_distinct) {
    if (!s || !st || !env_ids || !slots) return fail(SWARM_ERR_INVALID, "null argument");
    if (s->cfg.variant != SWARM_VARIANT_ASSEMBLY) return fail(SWARM_ERR_UNSUPPORTED, "the state store serves assembly handles");
    if (count < 1) return fail(SWARM_ERR_INVALID, "count must be >= 1");
    if (!same_config(s->cfg, st->cfg)) return fail(SWARM_ERR_INVALID, "the handle's configuration is not the store's");
    const int E = s->cfg.num_envs;
    std::vector<char> seen_env(envs_distinct ? E : 0), seen_slot(envs_distinct ? 0 : st->capacity);
    for (int k = 0; k < count; ++k) {
        if (env_ids[k] < 0 || env_ids[k] >= E) return fail(SWARM_ERR_INVALID, "env id out of range");
        if (slots[k] < 0 || slots[k] >= st->capacity) return fail(SWARM_ERR_INVALID, "slot out of range");
        char &seen = envs_distinct ? seen_env[env_ids[k]] : seen_slot[slots[k]];
        if (seen) return fail(SWARM_ERR_INVALID, envs_distinct ? "env ids must be distinct" : "slots must be distinct");
        seen = 1;
    }
    return SWARM_OK;
}

// k_state_copy over the pairs (env_ids[k], slots[k]), STATE_PAIRS_PER_LAUNCH per launch
static int state_copy(swarm_sim *s, swarm_state_store *st, bool save, const int32_t *env_ids, const int32_t *slots, int32_t count,
                      cudaStream_t stream) {
    CU_TRY(cudaSetDevice(s->cfg.device));
    StateCopyParams P;
    P.slots = st->d_slots; P.slot_bytes = st->slot_bytes; P.n_segs = 0; P.pad_ = 0;
    for (int g = 0; g < SEG_COUNT; ++g) {
        // a handle that has not stepped returns the prior of its current state: a_prior[last] is a_prior[pending]
        if (!st->row[g] || (!save && g == SEG_PRIOR_LAST && s->last == s->pending)) continue;
        StateSeg &S = P.seg[P.n_segs++];
        S.env = state_seg_base(s, g); S.row = st->row[g]; S.off = st->off[g]; S.shape_id = g == SEG_SHAPE; S.pad_ = 0;
    }
    for (int k0 = 0; k0 < count; k0 += STATE_PAIRS_PER_LAUNCH) {
        const int n = std::min(count - k0, STATE_PAIRS_PER_LAUNCH);
        // at most 32 KB of a slot per CTA, at least 4 KB, and at least two CTAs per SM when the launch carries few pairs
        const long long sb = st->slot_bytes;
        long long chunks = std::max((sb + 32767) / 32768, (2LL * st->n_sm + n - 1) / n);
        chunks = std::min(chunks, (sb + 4095) / 4096);
        P.chunk = ((sb + chunks - 1) / chunks + 15) & ~15LL;
        chunks = (sb + P.chunk - 1) / P.chunk;
        for (int k = 0; k < n; ++k) {
            const int slot = slots[k0 + k];
            const bool unmatched = !save && st->slot[slot].lib_fp != s->lib_fp;
            P.pair[k] = make_int2(env_ids[k0 + k], slot | (unmatched ? STATE_UNMATCHED : 0));
        }
        const dim3 grid((unsigned)chunks, (unsigned)n);
        if (save) k_state_copy<true><<<grid, STATE_THREADS, 0, stream>>>(P);
        else k_state_copy<false><<<grid, STATE_THREADS, 0, stream>>>(P);
        CU_TRY(cudaGetLastError());
        s->launches++;
    }
    return SWARM_OK;
}

extern "C" {

int swarm_state_store_create(const swarm_sim *s, int64_t capacity, swarm_state_store **out) {
    if (!s || !out) return fail(SWARM_ERR_INVALID, "null argument");
    if (s->cfg.variant != SWARM_VARIANT_ASSEMBLY) return fail(SWARM_ERR_UNSUPPORTED, "the state store serves assembly handles");
    if (capacity < 1 || capacity > INT32_MAX) return fail(SWARM_ERR_INVALID, "capacity must be in [1, 2^31)");
    CU_TRY(cudaSetDevice(s->cfg.device));
    int n_sm = 0;
    CU_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, s->cfg.device));
    const swarm_config &c = s->cfg;
    const long long n_a = c.n_a, osz = c.out_dtype == SWARM_F32 ? 4 : 8;
    long long row[SEG_COUNT] = {};
    row[SEG_P] = row[SEG_DP] = 2 * n_a * 8;
    row[SEG_GRID] = (long long)s->K.n_g_pad * 16; row[SEG_WBOX] = (long long)s->K.n_words * 16; row[SEG_FRAME] = 16;
    row[SEG_NG] = 4; row[SEG_THRESH] = 8; row[SEG_POSE] = sizeof(double4); row[SEG_SHAPE] = 4;
    row[SEG_NEAREST] = row[SEG_FLAGS] = 4 * n_a; row[SEG_NBR] = 4LL * TOPO * n_a;
    row[SEG_OBS] = (long long)s->K.obs_dim * n_a * osz; row[SEG_REWARD] = n_a * osz;
    if (c.want_prior) row[SEG_PRIOR_CUR] = row[SEG_PRIOR_LAST] = 2 * n_a * osz;
    if (c.emit_indices) { row[SEG_SENSED] = 4LL * c.num_obs_grid_max * n_a; row[SEG_OCC] = 4LL * c.num_occupied_grid_max * n_a; }
    swarm_state_store *st = new swarm_state_store();
    st->cfg = c; st->capacity = capacity; st->n_sm = n_sm;
    long long off = 0;
    for (int g = 0; g < SEG_COUNT; ++g) { st->row[g] = row[g]; st->off[g] = off; off += (row[g] + 15) & ~15LL; }
    st->slot_bytes = (off + 127) & ~127LL;
    st->slot.assign((size_t)capacity, swarm_state_store::Slot{});
    const cudaError_t e = cudaMalloc(&st->d_slots, (size_t)capacity * st->slot_bytes);
    if (e != cudaSuccess) {
        delete st;
        return fail(SWARM_ERR_CUDA, std::string("cudaMalloc of the state store failed: ") + cudaGetErrorString(e));
    }
    *out = st;
    return SWARM_OK;
}

int swarm_state_store_destroy(swarm_state_store *st) {
    if (!st) return SWARM_OK;
    cudaSetDevice(st->cfg.device);
    cudaFree(st->d_slots);
    delete st;
    return SWARM_OK;
}

int64_t swarm_state_slot_bytes(const swarm_state_store *st) { return st ? st->slot_bytes : 0; }

int swarm_state_save(swarm_sim *s, swarm_state_store *st, const int32_t *env_ids, const int32_t *slots, int32_t count, void *stream) {
    if (const int rc = state_check(s, st, env_ids, slots, count, false)) return rc;
    if (!s->observed) return fail(SWARM_ERR_INVALID, "swarm_state_save needs an observed handle");
    if (const int rc = state_copy(s, st, true, env_ids, slots, count, (cudaStream_t)stream)) return rc;
    for (int k = 0; k < count; ++k) {
        swarm_state_store::Slot &r = st->slot[slots[k]];
        r.filled = true;
        r.prior_valid = !s->prior_dirty;
        r.match = s->match.env[env_ids[k]];
        r.lib_fp = s->lib_fp;
    }
    return SWARM_OK;
}

int swarm_state_load(swarm_sim *s, swarm_state_store *st, const int32_t *slots, const int32_t *env_ids, int32_t count, void *stream) {
    if (const int rc = state_check(s, st, env_ids, slots, count, true)) return rc;
    for (int k = 0; k < count; ++k)
        if (!st->slot[slots[k]].filled) return fail(SWARM_ERR_INVALID, "slot is empty");
    if (!s->observed && count != s->cfg.num_envs)
        return fail(SWARM_ERR_INVALID, "a handle that was never observed can only be loaded as a whole");
    if (const int rc = state_copy(s, st, false, env_ids, slots, count, (cudaStream_t)stream)) return rc;
    for (int k = 0; k < count; ++k) {
        const swarm_state_store::Slot &r = st->slot[slots[k]];
        // the kernel wrote shape id -1 for a slot of another library: that env is unmatched
        s->match.set(env_ids[k], r.lib_fp == s->lib_fp ? r.match : MatchMirror::UNMATCHED);
        if (s->cfg.want_prior && !r.prior_valid) s->prior_dirty = true;     // the next step's k_prior gives the same values
    }
    s->observed = true;
    return SWARM_OK;
}

static int launch_step(swarm_sim *s, bool dyn, const void *act, int act_dtype, cudaStream_t st, const int32_t *env_list, int32_t count) {
    KParams K = s->K;
    K.act = act; K.act_f32 = (act_dtype == SWARM_F32);
    K.prior_next = s->buf.a_prior[dyn ? (1 - s->pending) : s->pending];
    K.env_list = env_list;
    const int ctas = env_list ? count : s->cfg.num_envs;
    const StepLaunch L = step_launch(s, dyn, swarm_fast_path(s));
    if (L.k1) { L.k1<<<ctas, s->nt, L.smem1, st>>>(K); s->launches++; }
    L.k2<<<ctas, s->nt, L.smem2, st>>>(K);
    s->launches++;
    CU_TRY(cudaGetLastError());
    return SWARM_OK;
}

static int flock_launch(swarm_sim *s, bool dyn, const void *act, int act_dtype, cudaStream_t st) {
    if (s->cfg.variant != SWARM_VARIANT_FLOCKING) return fail(SWARM_ERR_INVALID, "not a flocking handle (swarm_config.variant)");
    CU_TRY(cudaSetDevice(s->cfg.device));
    KParams K = s->K;
    K.act = act; K.act_f32 = (act_dtype == SWARM_F32);
    const bool f32 = s->cfg.out_dtype == SWARM_F32;
    // the assembly step's first half, unchanged (its shared memory, 8 KB at most, needs no raised limit)
    step_fn_t k1 = step_kernel(f32, dyn, false, 128, 1, 0, s->nt != 32);
    k1<<<s->cfg.num_envs, s->nt, s->smem1, st>>>(K);
    const double d_ref = 2.0 * s->cfg.r_avoid;
    if (f32) k_flock_reward<float><<<s->cfg.num_envs, s->nt, 0, st>>>(s->cfg.n_a, K.p, K.dp, K.nbr, K.T_avoid, d_ref, 1.0, 0.5, 0.5, K.periodic, K.half_w, K.half_h, (float *)s->buf.reward);
    else k_flock_reward<double><<<s->cfg.num_envs, s->nt, 0, st>>>(s->cfg.n_a, K.p, K.dp, K.nbr, K.T_avoid, d_ref, 1.0, 0.5, 0.5, K.periodic, K.half_w, K.half_h, (double *)s->buf.reward);
    CU_TRY(cudaGetLastError());
    s->launches += 2;
    s->observed = true;
    return SWARM_OK;
}

/* ---- predator-prey variant (stateless; VARIANTS.md 4) ---- */
int swarm_pp_obs_dim(const swarm_pp_config *c) {
    if (!c || c->struct_size != sizeof(swarm_pp_config)) return -1;
    return 4 * (2 * TOPO + (c->is_con_self_state ? 1 : 0));
}
static int pp_launch(const swarm_pp_config *c, const swarm_pp_buffers *b, bool dyn, const void *act, int act_dtype, uint64_t step,
                     cudaStream_t st) {
    if (!c || !b || c->struct_size != sizeof(swarm_pp_config) || b->struct_size != sizeof(swarm_pp_buffers))
        return fail(SWARM_ERR_INVALID, "swarm_pp: bad config / buffers (struct_size)");
    const int n = c->n_p + c->n_e;
    if (c->num_envs < 1 || c->n_p < 0 || c->n_e < 0 || n < 1 || n > 128) return fail(SWARM_ERR_UNSUPPORTED, "swarm_pp: 1 <= n_p + n_e <= 128");
    if (!b->p || !b->dp || !b->obs || !b->reward || !b->neighbor_index) return fail(SWARM_ERR_INVALID, "swarm_pp: null buffer");
    if (c->out_dtype != SWARM_F32 && c->out_dtype != SWARM_F64) return fail(SWARM_ERR_INVALID, "swarm_pp: out_dtype");
    for (int sgy : {c->strategy_p, c->strategy_e}) if (sgy < 0 || sgy > 3) return fail(SWARM_ERR_INVALID, "swarm_pp: strategy");
    if (dyn && (c->strategy_p == SWARM_PP_INPUT || c->strategy_e == SWARM_PP_INPUT) && !act) return fail(SWARM_ERR_INVALID, "swarm_pp: null actions");
    if (!(c->d_sen > 0) || !(c->size_a > 0) || !(c->dt > 0) || !(c->mass > 0)) return fail(SWARM_ERR_INVALID, "swarm_pp: d_sen, size_a, dt, mass must be positive");
    CU_TRY(cudaSetDevice(c->device));
    PPParams Q{};
    Q.n_p = c->n_p; Q.n_e = c->n_e; Q.self_state = c->is_con_self_state; Q.periodic = c->is_periodic; Q.billiards = c->billiards;
    Q.strat_p = c->strategy_p; Q.strat_e = c->strategy_e; Q.act_f32 = (act_dtype == SWARM_F32);
    Q.two_size = c->size_a + c->size_a; Q.size_a = c->size_a;
    Q.T_sen = thresh_lt(c->d_sen); Q.T_col = thresh_lt(Q.two_size);
    Q.k_ball = c->k_ball; Q.k_wall = c->k_wall; Q.c_wall = c->c_wall; Q.dt = c->dt; Q.vmax_p = c->vel_max_p; Q.vmax_e = c->vel_max_e; Q.mass = c->mass;
    Q.bx_min = c->boundary_pos[0]; Q.by_max = c->boundary_pos[1]; Q.bx_max = c->boundary_pos[2]; Q.by_min = c->boundary_pos[3];
    Q.half_w = (Q.bx_max - Q.bx_min) / 2.0; Q.half_h = (Q.by_max - Q.by_min) / 2.0;
    Q.p = b->p; Q.dp = b->dp; Q.act = act; Q.obs = b->obs; Q.reward = b->reward; Q.nbr = b->neighbor_index;
    Q.seed = c->seed; Q.step = step;
    const int nt = round32(n);
    const bool f32 = c->out_dtype == SWARM_F32;
    if (dyn) { if (f32) k_pp_step<float, true><<<c->num_envs, nt, 0, st>>>(Q); else k_pp_step<double, true><<<c->num_envs, nt, 0, st>>>(Q); }
    else { if (f32) k_pp_step<float, false><<<c->num_envs, nt, 0, st>>>(Q); else k_pp_step<double, false><<<c->num_envs, nt, 0, st>>>(Q); }
    CU_TRY(cudaGetLastError());
    return SWARM_OK;
}
int swarm_pp_observe(const swarm_pp_config *c, const swarm_pp_buffers *b, void *stream) {
    return pp_launch(c, b, false, nullptr, SWARM_F32, 0, (cudaStream_t)stream);
}
int swarm_pp_step(const swarm_pp_config *c, const swarm_pp_buffers *b, const void *act, int act_dtype, uint64_t step_index, void *stream) {
    if (act_dtype != SWARM_F32 && act_dtype != SWARM_F64) return fail(SWARM_ERR_INVALID, "swarm_pp: act_dtype");
    return pp_launch(c, b, true, act, act_dtype, step_index, (cudaStream_t)stream);
}

int swarm_flock_observe(swarm_sim *s, void *stream) {
    if (!s) return fail(SWARM_ERR_INVALID, "null handle");
    return flock_launch(s, false, nullptr, SWARM_F32, (cudaStream_t)stream);
}

int swarm_flock_step(swarm_sim *s, const void *act, int act_dtype, void *stream) {
    if (!s || !act) return fail(SWARM_ERR_INVALID, "null argument");
    if (act_dtype != SWARM_F32 && act_dtype != SWARM_F64) return fail(SWARM_ERR_INVALID, "bad act_dtype");
    return flock_launch(s, true, act, act_dtype, (cudaStream_t)stream);
}

int swarm_observe(swarm_sim *s, void *stream) {
    if (!s) return fail(SWARM_ERR_INVALID, "null handle");
    if (s->cfg.variant != SWARM_VARIANT_ASSEMBLY) return fail(SWARM_ERR_INVALID, "flocking handle: use swarm_flock_observe");
    CU_TRY(cudaSetDevice(s->cfg.device));
    int rc = launch_step(s, false, nullptr, SWARM_F32, (cudaStream_t)stream);
    if (rc != SWARM_OK) return rc;
    s->prior_dirty = false; s->observed = true;
    return SWARM_OK;
}

int swarm_step(swarm_sim *s, const void *act, int act_dtype, void *stream) {
    if (!s || !act) return fail(SWARM_ERR_INVALID, "null argument");
    if (act_dtype != SWARM_F32 && act_dtype != SWARM_F64) return fail(SWARM_ERR_INVALID, "bad act_dtype");
    if (s->cfg.variant != SWARM_VARIANT_ASSEMBLY) return fail(SWARM_ERR_INVALID, "flocking handle: use swarm_flock_step");
    if (!s->observed) return fail(SWARM_ERR_INVALID, "swarm_step before swarm_observe (reset)");
    cudaStream_t st = (cudaStream_t)stream;
    CU_TRY(cudaSetDevice(s->cfg.device));
    if (s->cfg.want_prior && s->prior_dirty) {
        // ENV:613-624 semantics: prior from the current p/dp/grid and the neighbour list of the last observation
        const int n_a = s->cfg.n_a;
        const int th = n_a < 256 ? round32(n_a) : 256;
        if (s->cfg.out_dtype == SWARM_F32)
            k_prior<float><<<s->cfg.num_envs, th, 0, st>>>(n_a, TOPO, s->K.p, s->K.dp, s->K.grid, s->K.n_g_pad, s->K.n_g,
                                                         s->K.in_thresh, s->K.nbr, s->K.r_avoid, (float *)s->buf.a_prior[s->pending]);
        else
            k_prior<double><<<s->cfg.num_envs, th, 0, st>>>(n_a, TOPO, s->K.p, s->K.dp, s->K.grid, s->K.n_g_pad, s->K.n_g,
                                                          s->K.in_thresh, s->K.nbr, s->K.r_avoid, (double *)s->buf.a_prior[s->pending]);
        CU_TRY(cudaGetLastError());
        s->launches++;
    }
    int rc = launch_step(s, true, act, act_dtype, st);
    if (rc != SWARM_OK) return rc;
    s->last = s->pending;
    s->pending = 1 - s->pending;
    s->prior_dirty = false;
    return SWARM_OK;
}

void *swarm_a_prior_ptr(swarm_sim *s) { return s ? s->buf.a_prior[s->last] : nullptr; }

int swarm_step_host(swarm_sim *s, const float *act_host, void *obs_host, void *reward_host, void *a_prior_host, void *stream) {
    if (!s || !act_host) return fail(SWARM_ERR_INVALID, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    CU_TRY(cudaSetDevice(s->cfg.device));
    const size_t E = s->cfg.num_envs, n = s->cfg.n_a;
    const size_t nact = E * 2 * n;
    if (const int rc = grow_staging(s->d_act, s->act_cap, nact)) return rc;
    CU_TRY(cudaMemcpyAsync(s->d_act, act_host, nact * sizeof(float), cudaMemcpyHostToDevice, st));
    int rc = swarm_step(s, s->d_act, SWARM_F32, stream);
    if (rc != SWARM_OK) return rc;
    const size_t osz = s->cfg.out_dtype == SWARM_F32 ? 4 : 8;
    if (obs_host) CU_TRY(cudaMemcpyAsync(obs_host, s->buf.obs, E * s->K.obs_dim * n * osz, cudaMemcpyDeviceToHost, st));
    if (reward_host) CU_TRY(cudaMemcpyAsync(reward_host, s->buf.reward, E * n * osz, cudaMemcpyDeviceToHost, st));
    if (a_prior_host) CU_TRY(cudaMemcpyAsync(a_prior_host, s->buf.a_prior[s->last], E * 2 * n * osz, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return SWARM_OK;
}

int swarm_fill_actions(swarm_sim *s, uint64_t seed, uint64_t step, uint64_t env_offset, float *act_dev, void *stream) {
    if (!s || !act_dev) return fail(SWARM_ERR_INVALID, "null argument");
    CU_TRY(cudaSetDevice(s->cfg.device));
    const long per_env = 2L * s->cfg.n_a, total = per_env * s->cfg.num_envs;
    const int blocks = (int)std::min<long>((total + 255) / 256, 148L * 16);
    k_fill_actions<<<blocks, 256, 0, (cudaStream_t)stream>>>(total, (int)per_env, seed, step, env_offset, act_dev);
    CU_TRY(cudaGetLastError());
    s->launches++;
    return SWARM_OK;
}

/* test hook: psi = _rho_cos_dec(z, 0, r) (CPP:1012-1020) of n HOST values through the device implementation */
int swarm_debug_rho(const double *z_host, int32_t n, double r, double *out_host) {
    if (!z_host || !out_host || n <= 0) return fail(SWARM_ERR_INVALID, "bad argument");
    double *d = nullptr;
    CU_TRY(cudaMalloc(&d, sizeof(double) * 2 * (size_t)n));
    cudaError_t e = cudaMemcpy(d, z_host, sizeof(double) * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) { k_debug_rho<<<(n + 255) / 256, 256>>>(d, n, r, d + n); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaMemcpy(out_host, d + n, sizeof(double) * n, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(SWARM_ERR_CUDA, std::string("swarm_debug_rho: ") + cudaGetErrorString(e));
    return SWARM_OK;
}

int64_t swarm_launch_count(const swarm_sim *s) { return s ? s->launches : 0; }

int swarm_kernel_geometry(const swarm_sim *s, int32_t *threads_per_cta, int32_t *smem_bytes, int32_t *ctas) {
    if (!s) return fail(SWARM_ERR_INVALID, "null handle");
    if (threads_per_cta) *threads_per_cta = s->nt;
    if (smem_bytes) *smem_bytes = (int32_t)s->smem;
    if (ctas) *ctas = s->cfg.num_envs;
    return SWARM_OK;
}

}  // extern "C"

// =====================================================================================================
// Legacy stateless entry points (HOST pointers).  Every call stages all its inputs in one pinned host buffer and moves them
// with ONE cudaMemcpy, runs its kernel(s), and brings all outputs back with ONE cudaMemcpy (the reference makes five such
// calls per env.step(); ten small synchronous copies per call were most of this path's time).  The packed cell list of the
// last grid is cached on the device: the reference passes the same grid_center for a whole episode.
// =====================================================================================================
namespace {

std::mutex g_legacy_mutex;

[[noreturn]] void legacy_die(const char *where, const std::string &msg) {
    fprintf(stderr, "[swarm_b200] %s: %s (no CPU fallback exists; aborting)\n", where, msg.c_str());
    abort();
}
#define LEG_TRY(where, expr)                                                             \
    do {                                                                                 \
        cudaError_t err__ = (expr);                                                      \
        if (err__ != cudaSuccess) legacy_die(where, std::string(#expr) + ": " + cudaGetErrorString(err__)); \
    } while (0)

// Device arena mirrored by a pinned host buffer: in() slots are filled on the host and uploaded together, out() slots are
// downloaded together and scattered to the caller's arrays.  Inputs first, then scratch / outputs (call order = layout order).
struct Xfer {
    static unsigned char *dev, *host; static size_t cap;
    const char *W; size_t off = 0, in_end = 0, out_begin = 0;
    struct Out { void *dst; size_t off, bytes; };
    std::vector<Out> outs;
    Xfer(size_t need, const char *where) : W(where) {
        need += 8192;
        if (need > cap) {
            if (dev) LEG_TRY(W, cudaFree(dev));
            if (host) LEG_TRY(W, cudaFreeHost(host));
            dev = host = nullptr; cap = 0;
            LEG_TRY(W, cudaMalloc(&dev, need));
            LEG_TRY(W, cudaHostAlloc(&host, need, cudaHostAllocDefault));
            cap = need;
        }
    }
    template <typename T> T *slot(size_t count) {
        off = (off + 255) & ~(size_t)255;
        T *ptr = reinterpret_cast<T *>(dev + off);
        off += count * sizeof(T);
        if (off > cap) legacy_die(W, "internal: legacy arena too small");
        return ptr;
    }
    template <typename T> T *in(const void *src, size_t count) {          // must precede every scratch() / out()
        T *d = slot<T>(count);
        memcpy(host + (reinterpret_cast<unsigned char *>(d) - dev), src, count * sizeof(T));
        in_end = off;
        return d;
    }
    void upload() { if (in_end) LEG_TRY(W, cudaMemcpy(dev, host, in_end, cudaMemcpyHostToDevice)); }
    template <typename T> T *scratch(size_t count) { return slot<T>(count); }
    template <typename T> T *out(void *dst, size_t count) {
        T *d = slot<T>(count);
        if (outs.empty()) out_begin = reinterpret_cast<unsigned char *>(d) - dev;
        outs.push_back({dst, (size_t)(reinterpret_cast<unsigned char *>(d) - dev), count * sizeof(T)});
        return d;
    }
    void download() {
        if (outs.empty()) return;
        LEG_TRY(W, cudaMemcpy(host + out_begin, dev + out_begin, off - out_begin, cudaMemcpyDeviceToHost));
        for (const Out &o : outs) memcpy(o.dst, host + o.off, o.bytes);
    }
};
unsigned char *Xfer::dev = nullptr, *Xfer::host = nullptr; size_t Xfer::cap = 0;

size_t al(size_t b) { return (b + 255) & ~(size_t)255; }

// packed cell list (+ word boxes, frame, n_g, in-shape threshold) of the most recent grid_center, kept on the device
struct GridCache {
    std::vector<double> host; int n_g = -1, n_g_pad = 0; double l_cell = 0.0; size_t cap_cells = 0;
    unsigned char *block = nullptr;          // [src 2*n_g f64 | cells n_g_pad double2 | boxes | frame | n_g | thr]
    double *src = nullptr; double2 *cells = nullptr; float4 *box = nullptr; double *frame = nullptr; int *d_ng = nullptr; double *d_thr = nullptr;
} g_grid;

void legacy_grid(const char *W, const double *grid_center, int n_g, double l_cell) {
    const int n_g_pad = round32(n_g);
    const bool same = g_grid.n_g == n_g && g_grid.l_cell == l_cell && memcmp(g_grid.host.data(), grid_center, sizeof(double) * 2 * (size_t)n_g) == 0;
    if (same) return;
    if ((size_t)n_g_pad > g_grid.cap_cells) {
        if (g_grid.block) LEG_TRY(W, cudaFree(g_grid.block));
        const size_t bytes = al(2 * (size_t)n_g_pad * 8) + al((size_t)n_g_pad * 16) + al((size_t)n_g_pad / 32 * 16) + 4 * 256;
        LEG_TRY(W, cudaMalloc(&g_grid.block, bytes));
        g_grid.cap_cells = n_g_pad;
        unsigned char *q = g_grid.block;
        g_grid.src = reinterpret_cast<double *>(q); q += al(2 * (size_t)n_g_pad * 8);
        g_grid.cells = reinterpret_cast<double2 *>(q); q += al((size_t)n_g_pad * 16);
        g_grid.box = reinterpret_cast<float4 *>(q); q += al((size_t)n_g_pad / 32 * 16);
        g_grid.frame = reinterpret_cast<double *>(q); q += 256;
        g_grid.d_ng = reinterpret_cast<int *>(q); q += 256;
        g_grid.d_thr = reinterpret_cast<double *>(q);
    }
    const double thr = in_shape_thresh(l_cell);
    LEG_TRY(W, cudaMemcpy(g_grid.src, grid_center, sizeof(double) * 2 * (size_t)n_g, cudaMemcpyHostToDevice));
    LEG_TRY(W, cudaMemcpy(g_grid.d_ng, &n_g, 4, cudaMemcpyHostToDevice));
    LEG_TRY(W, cudaMemcpy(g_grid.d_thr, &thr, 8, cudaMemcpyHostToDevice));
    k_pack_grid<<<1, 128>>>(g_grid.src, 2L * n_g, g_grid.d_ng, n_g_pad, g_grid.cells, g_grid.box, g_grid.frame, PoseArgs{});
    LEG_TRY(W, cudaGetLastError());
    g_grid.host.assign(grid_center, grid_center + 2 * (size_t)n_g);
    g_grid.n_g = n_g; g_grid.n_g_pad = n_g_pad; g_grid.l_cell = l_cell;
}

}  // namespace

extern "C" {

void _get_observation(double *p, double *dp, double *heading, double *obs, double *boundary_pos, double *grid_center,
                      int *neighbor_index, int *in_flags, int *sensed_index, int *occupied_index, double d_sen,
                      double r_avoid, double l_cell, double Vel_max, int topo_nei_max, int num_obs_grid_max,
                      int num_occupied_grid_max, int n_a, int n_g, int obs_dim_agent, int dim, bool *condition) {
    const char *W = "_get_observation";
    (void)heading; (void)Vel_max;
    if (dim != 2 || topo_nei_max != TOPO) legacy_die(W, "only dim == 2 and topo_nei_max == 6 are supported");
    if (!condition[1]) legacy_die(W, "only Cartesian dynamics are implemented");
    if (n_a > 1024 || n_a <= 0 || n_g <= 0) legacy_die(W, "n_a must be in [1,1024] and n_g positive");
    std::lock_guard<std::mutex> lock(g_legacy_mutex);
    KParams K; memset(&K, 0, sizeof(K));
    fill_constants(K, n_a, n_g, num_obs_grid_max, num_occupied_grid_max, condition[2], false, false, condition[0], d_sen, r_avoid,
                   0.035, 30.0, 100.0, 5.0, 0.1, 0.8, 1.0, boundary_pos);
    if (K.obs_dim != obs_dim_agent) legacy_die(W, "obs_dim_agent does not match 2*2*(6+1+self)+2*num_obs_grid_max");
    K.E = 1;
    const int nt = round32(n_a);
    const size_t smem = step_smem_bytes(nt, K.n_words, true, num_obs_grid_max);
    const size_t n_obs = (size_t)K.obs_dim * n_a;
    legacy_grid(W, grid_center, n_g, l_cell);
    Xfer X(al(4 * (size_t)n_a * 8) * 2 + al(n_obs * 8) + al((size_t)n_a * 8 * 3) + al((size_t)n_a * TOPO * 4) + al((size_t)n_a * 8) +
           al((size_t)n_a * num_obs_grid_max * 4) + al((size_t)n_a * num_occupied_grid_max * 4) + 16 * 256, W);
    double *d_p = X.in<double>(p, 2 * (size_t)n_a), *d_dp = X.in<double>(dp, 2 * (size_t)n_a);
    X.upload();
    double *d_rew = X.scratch<double>(n_a), *d_prior = X.scratch<double>(2 * (size_t)n_a);
    int *d_near = X.scratch<int>(n_a);
    double *d_obs = X.out<double>(obs, n_obs);
    int *d_nbr = X.out<int>(neighbor_index, (size_t)n_a * TOPO), *d_inf = X.out<int>(in_flags, n_a);
    int *d_sidx = X.out<int>(sensed_index, (size_t)n_a * num_obs_grid_max), *d_occ = X.out<int>(occupied_index, (size_t)n_a * num_occupied_grid_max);
    LEG_TRY(W, cudaMemset(d_near, 0, (size_t)n_a * 4));
    K.wbox = g_grid.box; K.frame = g_grid.frame;
    K.p = d_p; K.dp = d_dp; K.grid = g_grid.cells; K.n_g = g_grid.d_ng; K.in_thresh = g_grid.d_thr;
    K.obs = d_obs; K.reward = d_rew; K.prior_next = d_prior;
    K.nbr = d_nbr; K.in_flags = d_inf; K.nearest = d_near; K.sensed = d_sidx; K.occupied = d_occ;
    step_fn_t f = step_kernel(false, false, true, nt <= 128 ? 128 : 1024, 0);
    LEG_TRY(W, raise_smem_limit((const void *)f, smem));
    f<<<1, nt, smem>>>(K);
    LEG_TRY(W, cudaGetLastError());
    X.download();
}

void _get_reward(double *p, double *dp, double *heading, double *act, double *reward, double *boundary_pos,
                 double *grid_center, int *neighbor_index, int *in_flags, int *sensed_index, int *occupied_index,
                 double d_sen, double r_avoid, double l_cell, int topo_nei_max, int num_obs_grid_max,
                 int num_occupied_grid_max, int n_a, int n_g, int dim, bool *condition, bool *is_collide_b2b,
                 bool *is_collide_b2w, double *coefficients) {
    const char *W = "_get_reward";
    (void)dp; (void)heading; (void)act; (void)occupied_index;
    (void)num_occupied_grid_max; (void)is_collide_b2b; (void)is_collide_b2w; (void)coefficients;
    if (dim != 2) legacy_die(W, "only dim == 2 is supported");
    std::lock_guard<std::mutex> lock(g_legacy_mutex);
    legacy_grid(W, grid_center, n_g, l_cell);             // k_legacy_reward reads the [2][n_g] copy kept beside the packed cells
    Xfer X(al(2 * (size_t)n_a * 8) + al((size_t)n_a * topo_nei_max * 4) + al((size_t)n_a * 4) +
           al((size_t)n_a * num_obs_grid_max * 4) + al((size_t)n_a * 8) + 8 * 256, W);
    double *d_p = X.in<double>(p, 2 * (size_t)n_a);
    int *d_nbr = X.in<int>(neighbor_index, (size_t)n_a * topo_nei_max), *d_inf = X.in<int>(in_flags, n_a);
    int *d_sidx = X.in<int>(sensed_index, (size_t)n_a * num_obs_grid_max);
    X.upload();
    double *d_r = X.out<double>(reward, n_a);
    k_legacy_reward<<<(n_a + 127) / 128, 128>>>(d_p, g_grid.src, d_nbr, d_inf, d_sidx, n_a, n_g, topo_nei_max, num_obs_grid_max,
                                               d_sen, r_avoid, condition[3], condition[4], condition[0],
                                               (boundary_pos[2] - boundary_pos[0]) / 2.0, (boundary_pos[1] - boundary_pos[3]) / 2.0, d_r);
    LEG_TRY(W, cudaGetLastError());
    X.download();
}

void _sf_b2b_all(double *p, double *sf_b2b, double *d_b2b_edge, bool *is_collide_b2b, double *boundary_pos,
                 double *d_b2b_center, int n_a, int dim, double k_ball, bool is_periodic) {
    const char *W = "_sf_b2b_all";
    if (dim != 2) legacy_die(W, "only dim == 2 is supported");
    std::lock_guard<std::mutex> lock(g_legacy_mutex);
    const size_t nn = (size_t)n_a * n_a;
    Xfer X(al(2 * (size_t)n_a * 8) * 2 + al(nn * 8) * 2 + al(nn) + 8 * 256, W);
    double *d_p = X.in<double>(p, 2 * (size_t)n_a);
    double *d_e = X.in<double>(d_b2b_edge, nn), *d_c = X.in<double>(d_b2b_center, nn);
    unsigned char *d_col = X.in<unsigned char>(is_collide_b2b, nn);
    X.upload();
    double *d_sf = X.out<double>(sf_b2b, 2 * (size_t)n_a);
    k_legacy_sf_b2b<<<(n_a + 127) / 128, 128>>>(d_p, d_e, d_col, d_c, n_a, k_ball, is_periodic ? 1 : 0,
                                               (boundary_pos[2] - boundary_pos[0]) / 2.0, (boundary_pos[1] - boundary_pos[3]) / 2.0, d_sf);
    LEG_TRY(W, cudaGetLastError());
    X.download();
}

void _get_dist_b2w(double *p, double *r, double *d_b2w, bool *isCollision, int dim, int n_a, double *boundary_pos) {
    const char *W = "_get_dist_b2w";
    if (dim != 2) legacy_die(W, "only dim == 2 is supported");
    std::lock_guard<std::mutex> lock(g_legacy_mutex);
    Xfer X(al(2 * (size_t)n_a * 8) + al((size_t)n_a * 8) + al(4 * (size_t)n_a * 8) + al(4 * (size_t)n_a) + al(32) + 8 * 256, W);
    double *d_p = X.in<double>(p, 2 * (size_t)n_a), *d_r = X.in<double>(r, n_a), *d_bp = X.in<double>(boundary_pos, 4);
    X.upload();
    double *d_d = X.out<double>(d_b2w, 4 * (size_t)n_a);
    unsigned char *d_col = X.out<unsigned char>(isCollision, 4 * (size_t)n_a);
    k_legacy_b2w<<<(n_a + 127) / 128, 128>>>(d_p, d_r, d_bp, n_a, d_d, d_col);
    LEG_TRY(W, cudaGetLastError());
    X.download();
}

void calculateActionPrior(double *p, double *dp, double *a_prior, double *grid_center, int *neighbor_index, double d_sen,
                          double r_avoid, double l_cell, int topo_nei_max, int n_a, int n_g, int dim) {
    const char *W = "calculateActionPrior";
    (void)d_sen;
    if (dim != 2) legacy_die(W, "only dim == 2 is supported");
    std::lock_guard<std::mutex> lock(g_legacy_mutex);
    legacy_grid(W, grid_center, n_g, l_cell);
    Xfer X(al(2 * (size_t)n_a * 8) * 3 + al((size_t)n_a * topo_nei_max * 4) + 12 * 256, W);
    double *d_p = X.in<double>(p, 2 * (size_t)n_a), *d_dp = X.in<double>(dp, 2 * (size_t)n_a);
    int *d_nbr = X.in<int>(neighbor_index, (size_t)n_a * topo_nei_max);
    X.upload();
    double *d_out = X.out<double>(a_prior, 2 * (size_t)n_a);
    k_prior<double><<<1, n_a < 256 ? round32(n_a) : 256>>>(n_a, topo_nei_max, d_p, d_dp, g_grid.cells, g_grid.n_g_pad, g_grid.d_ng, g_grid.d_thr,
                                                           d_nbr, r_avoid, d_out);
    LEG_TRY(W, cudaGetLastError());
    X.download();
}

}  // extern "C"
