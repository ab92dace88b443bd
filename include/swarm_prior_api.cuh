/*
 * swarm_prior_api.cuh — the program interface of prior policies (DESIGN.md §12).
 *
 * A prior policy is the `robotPolicy` of the reference (CPP:1121-1196): a function of one agent's view of its env that
 * returns a 2-D action.  MADDPG regularises the learned policy towards it (the fifth output of step(), ENV:605-624).
 * A program replaces the built-in prior without rebuilding the library: the caller writes exactly one function
 *
 *     #include "swarm_prior_api.cuh"
 *     __device__ void robot_policy(const swarm_agent &a, double out[2]) { ... }
 *
 * and swarm_prior_compile (include/swarm_b200.h) compiles it at run time for sm_100a with NVRTC.  The library supplies this
 * header: the source needs no file path and no other include (there are no system headers; sqrt, fabs, fmin, fmax and the
 * other CUDA math functions are built in).
 *
 * Arithmetic: the program is compiled with --fmad=false and NVRTC's IEEE division and square root, the same contract as the
 * library's kernels: every fp64 operation is rounded on its own, so `x * x + y * y` is two products and a sum, exactly what an
 * x86-64 build of the reference computes.  A program that restates the reference's arithmetic in the reference's order
 * reproduces its prior bit for bit (marl_llm_b200/priors/reference_prior.cu does).
 *
 * What `a` holds (read-only) is the state BEFORE the step that returns the prior, the state ENV:613-624 hands to
 * calculateActionPrior: the positions and velocities, the target grid, and the neighbour list of the last observation.
 * out[0], out[1] are the x and y components; the library stores them as they are (a_prior in the handle's output dtype,
 * or fp64 actions), so a program clamps its result itself, as the reference does (CPP:1192-1193).
 *
 * Units and frames are the reference's: positions in the arena [boundary[0], boundary[2]] x [boundary[3], boundary[1]],
 * velocities per unit time, all fp64.  Accessors clamp their index into range, so a stray index reads some agent or cell of
 * the same env, never another env's memory.
 */
#ifndef SWARM_PRIOR_API_CUH
#define SWARM_PRIOR_API_CUH

#define SWARM_PRIOR_TOPO 6          /* ENV:34 topo_nei_max: the neighbour list holds at most 6 agents */

/* A 2-D vector (x, y). */
struct swarm_xy {
    double x, y;
};

/* Kernel parameters of the entry points below; filled by the library (its host code includes this header for the layout). */
struct swarm_prior_args {
    int n_a, n_g_pad;                  /* agents per env; cells per grid row (n_g rounded up to 32) */
    int stored;                        /* 1: nearest cell / in-shape flag from the last observation; 0: scanned here */
    int pad_;
    const double *p, *dp;              /* [E][2][n_a] */
    const double *grid;                /* [E][n_g_pad][2] (x, y) */
    const int *n_g;                    /* [E] */
    const double *in_thresh;           /* [E] squared in-shape radius threshold */
    const int *nbr;                    /* [E][n_a][6] neighbour ids, -1 = empty */
    const int *nearest;                /* [E][n_a] nearest cell of the last observation */
    const int *in_flags;               /* [E][n_a] bit 0: in the shape at the last observation */
    double d_sen, r_avoid, size_a, vel_max, dt;
    double boundary[4];
    void *out;                         /* [E][2][n_a] f32 or f64 */
    const int *env_ids;                /* CTA b serves env env_ids[b] (a population's group); NULL: env b */
};

#ifdef __CUDACC_RTC__

/* One agent of one env, in the pre-step state.  Field names follow the reference; each cites where the reference takes it. */
struct swarm_agent {
    int env;                           /* env index in the batch (0 .. E-1) */
    int id;                            /* agent index i (0 .. n_a-1), the `i` of robotPolicy (CPP:1121) */
    int n_a;                           /* agents in the env (ENV:99) */
    double x, y;                       /* p[:, i], position (CPP:1125-1126) */
    double vx, vy;                     /* dp[:, i], velocity (CPP:1127-1128) */
    bool in_shape;                     /* in_flag: the nearest cell is within sqrt(2) * l_cell / 2 (CPP:889) */
    int nearest;                       /* index of the nearest cell: the first minimum of the distances (CPP:869-887) */
    double cell_x, cell_y;             /* that cell's position, the target when !in_shape (CPP:891-897, 1102, 1136-1140) */
    int count;                         /* neighbours listed (0 .. 6): neighbor(0 .. count-1), nearest first (CPP:628-698) */
    /* constants of the env (ENV:28-60, 124, 193-196) */
    double d_sen;                      /* sensing radius */
    double r_avoid;                    /* avoidance radius (ENV:124), the `r_avoid` of CPP:1166 */
    double size_a;                     /* agent radius */
    double vel_max;                    /* speed cap per axis (ENV:647) */
    double dt;                         /* time step (ENV:646) */
    double in_thresh;                  /* in_shape <=> (squared distance to the nearest cell) < in_thresh (CPP:889, squared) */
    double boundary[4];                /* xmin, ymax, xmax, ymin (ENV:193-196) */

    /* agent id of neighbour q of the list, list order (neighbor_index, CPP:1151-1160; q clamped into 0 .. count-1); -1 when
     * count == 0.  The observation writes the ids nearest first and -1 after the last one. */
    __device__ int neighbor(int q) const {
        if (count <= 0) return -1;
        q = q < 0 ? 0 : (q >= count ? count - 1 : q);
        return nbr_[q];
    }
    /* position / velocity of any agent j of this env (j clamped into 0 .. n_a-1): p[:, j], dp[:, j] */
    __device__ swarm_xy pos(int j) const { j = clamp_(j, n_a); swarm_xy r; r.x = p_[j]; r.y = p_[n_a + j]; return r; }
    __device__ swarm_xy vel(int j) const { j = clamp_(j, n_a); swarm_xy r; r.x = dp_[j]; r.y = dp_[n_a + j]; return r; }
    /* number of target cells n_g of this env (ENV:163), and cell k (k clamped into 0 .. n_g-1): grid_center[:, k] */
    __device__ int n_g() const { return n_g_; }
    __device__ swarm_xy cell(int k) const { k = clamp_(k, n_g_); swarm_xy r; r.x = grid_[2 * k]; r.y = grid_[2 * k + 1]; return r; }

    /* the library's part of the view */
    const double *p_, *dp_, *grid_;
    const int *nbr_;
    int n_g_;
    __device__ static int clamp_(int k, int n) { return k < 0 ? 0 : (k >= n ? n - 1 : k); }
};

#endif
#endif /* SWARM_PRIOR_API_CUH */

/*
 * Entry points.  swarm_prior_compile appends `#define SWARM_PRIOR_ENTRY` and `#include "swarm_prior_api.cuh"` to the program,
 * so they follow the program's robot_policy.  One CTA per env, threads striding over its agents (the geometry of k_prior); with
 * env_ids, CTA b serves env env_ids[b] and the others are left as they are (a population runs each program on its own envs):
 *   swarm_prior_f32 / swarm_prior_f64   a_prior of the handle, [E][2][n_a] in the output dtype
 *   swarm_prior_actions                  actions [E][2][n_a] f64
 * The nearest cell is the one the last observation stored when that observation is of the current state and grid (stored =
 * 1), otherwise the first minimum of the squared distances over the env's cells, the scan k_prior does.
 */
#if defined(__CUDACC_RTC__) && defined(SWARM_PRIOR_ENTRY) && !defined(SWARM_PRIOR_ENTRY_DONE)
#define SWARM_PRIOR_ENTRY_DONE

template <typename OUT>
__device__ void swarm_prior_run_(const swarm_prior_args &A) {
    const int e = A.env_ids ? A.env_ids[blockIdx.x] : (int)blockIdx.x, n_a = A.n_a;
    const double *pe = A.p + (size_t)e * 2 * n_a, *dpe = A.dp + (size_t)e * 2 * n_a;
    const double *g = A.grid + (size_t)e * A.n_g_pad * 2;
    const int n_g = A.n_g[e];
    const double thr = A.in_thresh[e];
    OUT *out = reinterpret_cast<OUT *>(A.out) + (size_t)e * 2 * n_a;
    for (int i = threadIdx.x; i < n_a; i += blockDim.x) {
        swarm_agent a;
        a.env = e; a.id = i; a.n_a = n_a;
        a.x = pe[i]; a.y = pe[n_a + i]; a.vx = dpe[i]; a.vy = dpe[n_a + i];
        int bc = 0;
        if (A.stored) {
            bc = A.nearest[(size_t)e * n_a + i];
            bc = bc < 0 ? 0 : (bc >= n_g ? n_g - 1 : bc);
            a.in_shape = (A.in_flags[(size_t)e * n_a + i] & 1) != 0;
        } else {
            double best = __longlong_as_double(0x7ff0000000000000LL);
            for (int c = 0; c < n_g; ++c) {
                const double dx = g[2 * c] - a.x, dy = g[2 * c + 1] - a.y;
                const double s = dx * dx + dy * dy;
                if (s < best) { best = s; bc = c; }
            }
            a.in_shape = best < thr;
        }
        a.nearest = bc; a.cell_x = g[2 * bc]; a.cell_y = g[2 * bc + 1];
        a.nbr_ = A.nbr + ((size_t)e * n_a + i) * SWARM_PRIOR_TOPO;
        a.count = 0;
        while (a.count < SWARM_PRIOR_TOPO && a.nbr_[a.count] >= 0) a.count++;
        a.d_sen = A.d_sen; a.r_avoid = A.r_avoid; a.size_a = A.size_a; a.vel_max = A.vel_max; a.dt = A.dt; a.in_thresh = thr;
        for (int k = 0; k < 4; ++k) a.boundary[k] = A.boundary[k];
        a.p_ = pe; a.dp_ = dpe; a.grid_ = g; a.n_g_ = n_g;
        double o[2] = {0.0, 0.0};
        robot_policy(a, o);
        out[i] = (OUT)o[0];
        out[n_a + i] = (OUT)o[1];
    }
}

extern "C" __global__ void swarm_prior_f32(const swarm_prior_args A) { swarm_prior_run_<float>(A); }
extern "C" __global__ void swarm_prior_f64(const swarm_prior_args A) { swarm_prior_run_<double>(A); }
extern "C" __global__ void swarm_prior_actions(const swarm_prior_args A) { swarm_prior_run_<double>(A); }

#endif
