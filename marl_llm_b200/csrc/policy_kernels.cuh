// policy_kernels.cuh — the rollout policy on the device (SURVEY.md §8 f1): MADDPG.step() of the reference
// (marl_llm/algorithm/algorithms/maddpg.py:72-87 -> utils/agents.py:69-96 -> utils/networks.py:33-44) evaluated for every
// agent of every env straight from the simulator's observation layout.
//
//   obs [E][K0][n_a] f32 (feature-major, what k_step writes)  ->  act [E][A][n_a] f32 (what k_step reads)
//   h1 = leaky_relu(W1 obs + b1); h2 = leaky_relu(W2 h1 + b2); h3 = leaky_relu(W3 h2 + b3); a = tanh(W4 h3 + b4)
//   explore (agents.py:85-93): a += scale * N(0,1), clamp to [-1,1]  |  or a = U(-1,1) for the whole batch (epsilon branch)
//
// k_policy_mlp is the exact-fp32 path: plain FFMA, fp32 accumulation in a fixed k-ascending order (deterministic; agrees
// with torch's fp32 Linear to rounding).  A "column" is one agent; a CTA owns POL_M columns, keeps their activations in
// shared memory as [k][column] for all four layers (nothing but obs is read from and nothing but act written to HBM),
// and streams the (L2-resident, pre-transposed, zero-padded) weights through a double-buffered cp.async ring.
// Each thread accumulates a 6 (outputs) x 8 (columns) register tile: 48 FFMA per 3 + 2 shared-memory vector loads.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <stdint.h>

namespace swarm {

constexpr int POL_M = 64;        // columns (agents) per CTA
constexpr int POL_HP = 192;      // padded hidden width and padded input width (reference: hidden 180, obs 192)
constexpr int POL_KC = 16;       // k rows per weight chunk
constexpr int POL_THREADS = 256; // 32 output tiles of 6  x  8 column tiles of 8
constexpr int POL_AMAX = 8;      // largest action dimension

struct PolicyParams {
    const float *obs; float *act; float *log_pi;        // log_pi [E][1][n_a] or NULL
    float *rows_out;             // optional [E*n_a][K0]: every agent's observation as one row (replay storage for free), or NULL
    int obs_am;                  // obs is agent-major [E*n_a][K0] (k_step with SWARM_OBS_AGENT_MAJOR) instead of [E][K0][n_a]
    long n_cols;                 // E * n_a
    int n_a, K0, A;              // agents per env, observation features (<= POL_HP), action dimension (<= POL_AMAX)
    const float *Wt[3];          // [POL_HP][POL_HP] transposed weights Wt[k][n] of the three hidden layers, zero-padded
    const float *b[3];           // [POL_HP] biases, zero-padded
    const float *W4;             // [A][POL_HP] output layer (row-major like torch), zero-padded
    const float *b4;             // [A]
    float slope;                 // leaky_relu negative slope (torch default 0.01, networks.py:11)
    int explore;                 // 0 none | 1 gaussian | 2 uniform (agents.py:85-93)
    float scale;                 // noise scale (utils/noise.py:30)
    uint64_t seed, step;         // keys of the counter-based generator
};

__device__ __forceinline__ uint64_t pol_mix64(uint64_t seed, uint64_t a, uint64_t b, uint64_t k) {
    uint64_t z = seed * 0x9E3779B97F4A7C15ull + a * 0xBF58476D1CE4E5B9ull + b * 0x94D049BB133111EBull + k * 0xD6E8FEB86659FD93ull;
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    z ^= z >> 31;
    return z;
}
// component j of column col's exploration draws (agents.py:85-93), shared by every policy kernel: a unit-variance
// Gaussian (Box-Muller; the noise is this times P.scale) and the epsilon branch's uniform action in [-1, 1)
__device__ __forceinline__ float pol_gauss(const PolicyParams &P, long col, int j) {
    const uint64_t r = pol_mix64(P.seed, P.step, (uint64_t)col, (uint64_t)j);
    const float u1 = ((float)(r >> 40) + 1.0f) * (1.0f / 16777216.0f);          // (0, 1]
    const float u2 = (float)((r >> 16) & 0xffffffu) * (1.0f / 16777216.0f);     // [0, 1)
    return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}
__device__ __forceinline__ float pol_uniform(const PolicyParams &P, long col, int j) {
    const uint64_t r = pol_mix64(P.seed, P.step, (uint64_t)col, (uint64_t)j);
    return (float)(r >> 40) * (2.0f / 16777216.0f) - 1.0f;
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__global__ void __launch_bounds__(POL_THREADS, 1) k_policy_mlp(const PolicyParams P) {
    extern __shared__ __align__(16) float psm[];
    float *hA = psm;                               // [POL_HP][POL_M] activations (ping)
    float *hB = hA + POL_HP * POL_M;               // [POL_HP][POL_M] activations (pong)
    float *wbuf = hB + POL_HP * POL_M;             // [2][POL_KC][POL_HP] weight chunks
    const int tid = threadIdx.x;
    const long c0 = (long)blockIdx.x * POL_M;      // first column of this CTA
    const int n_a = P.n_a;

    // ---- observation tile: hA[k][c] = obs[e][k][a], column c0 + c = e * n_a + a; rows K0..POL_HP-1 and dead columns = 0
    for (int idx = tid; idx < POL_HP * POL_M; idx += POL_THREADS) {
        const int k = idx / POL_M, c = idx - k * POL_M;
        const long col = c0 + c;
        float v = 0.f;
        if (k < P.K0 && col < P.n_cols) {
            const long e = col / n_a; const int a = (int)(col - e * n_a);
            v = P.obs_am ? P.obs[col * P.K0 + k] : P.obs[(e * P.K0 + k) * n_a + a];
            if (P.rows_out) P.rows_out[col * P.K0 + k] = v;
        }
        hA[idx] = v;
    }

    // this thread's 6 x 8 output tile: outputs n0..n0+5, columns a0..a0+3 and a0+32..a0+35 (the 8 lanes sharing n0 read one
    // contiguous 128-byte line per vector load: conflict-free)
    const int n0 = (tid >> 3) * 6, a0 = (tid & 7) * 4;
    float *hin = hA, *hout = hB;
#pragma unroll 1
    for (int layer = 0; layer < 3; ++layer) {
        const float *Wt = P.Wt[layer];
        float acc[6][8];
#pragma unroll
        for (int r = 0; r < 6; ++r)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
        // chunk 0 in flight; the __syncthreads below also covers the activation tile written above / by the last layer
        for (int q = tid; q < POL_KC * POL_HP / 4; q += POL_THREADS) cp_async16(wbuf + q * 4, Wt + q * 4);
        cp_async_commit();
#pragma unroll 1
        for (int ch = 0; ch < POL_HP / POL_KC; ++ch) {
            if (ch + 1 < POL_HP / POL_KC) {
                float *dst = wbuf + ((ch + 1) & 1) * POL_KC * POL_HP;
                const float *src = Wt + (size_t)(ch + 1) * POL_KC * POL_HP;
                for (int q = tid; q < POL_KC * POL_HP / 4; q += POL_THREADS) cp_async16(dst + q * 4, src + q * 4);
                cp_async_commit();
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncthreads();                                   // chunk ch (and the input activations) visible to all
            const float *w = wbuf + (ch & 1) * POL_KC * POL_HP;
#pragma unroll 4
            for (int kk = 0; kk < POL_KC; ++kk) {
                const int k = ch * POL_KC + kk;
                const float2 w01 = *reinterpret_cast<const float2 *>(w + kk * POL_HP + n0);
                const float2 w23 = *reinterpret_cast<const float2 *>(w + kk * POL_HP + n0 + 2);
                const float2 w45 = *reinterpret_cast<const float2 *>(w + kk * POL_HP + n0 + 4);
                const float4 x0 = *reinterpret_cast<const float4 *>(hin + k * POL_M + a0);
                const float4 x1 = *reinterpret_cast<const float4 *>(hin + k * POL_M + a0 + 32);
                const float wr[6] = {w01.x, w01.y, w23.x, w23.y, w45.x, w45.y};
                const float xr[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
                for (int r = 0; r < 6; ++r)
#pragma unroll
                    for (int c = 0; c < 8; ++c) acc[r][c] = fmaf(wr[r], xr[c], acc[r][c]);
            }
            __syncthreads();                                   // everyone is done with buffer ch & 1 before it is refilled
        }
        const float *bias = P.b[layer];
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            const float bn = __ldg(bias + n0 + r);
            float o[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) { const float v = acc[r][c] + bn; o[c] = v > 0.f ? v : v * P.slope; }   // F.leaky_relu
            *reinterpret_cast<float4 *>(hout + (n0 + r) * POL_M + a0) = make_float4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<float4 *>(hout + (n0 + r) * POL_M + a0 + 32) = make_float4(o[4], o[5], o[6], o[7]);
        }
        float *t = hin; hin = hout; hout = t;
    }
    __syncthreads();                                           // h3 complete

    // ---- output layer + tanh + exploration: one (column, action component) per thread
    for (int idx = tid; idx < POL_M * P.A; idx += POL_THREADS) {
        const int j = idx / POL_M, c = idx - j * POL_M;
        const long col = c0 + c;
        if (col >= P.n_cols) continue;
        const float *w4 = P.W4 + (size_t)j * POL_HP;
        float s = 0.f;
#pragma unroll 4
        for (int k = 0; k < POL_HP; ++k) s = fmaf(__ldg(w4 + k), hin[k * POL_M + c], s);
        float a = tanhf(s + __ldg(P.b4 + j));                  // networks.py:29,43 (constrain_out)
        if (P.explore == 1) a = fminf(fmaxf(a + pol_gauss(P, col, j) * P.scale, -1.f), 1.f);   // agents.py:90-93, clamp
        else if (P.explore == 2) a = pol_uniform(P, col, j);  // agents.py:86-88: uniform action for the whole batch
        const long e = col / n_a; const int ag = (int)(col - e * n_a);
        P.act[(e * P.A + j) * n_a + ag] = a;
        if (P.log_pi) {
            // agents.py:82,88,91 + noise.py:32-37; the components of one column live in lanes POL_M apart: recompute them
            float lp = 0.f;
            if (P.explore == 2) lp = -(float)P.A * 0.69314718056f;
            else if (P.explore == 1 && j == 0) {
                float q = 0.f;
                for (int jj = 0; jj < P.A; ++jj) {
                    const float g = pol_gauss(P, col, jj);
                    q += g * g;
                }
                lp = -0.5f * q - (float)P.A * logf(P.scale * 2.50662827463f);
            }
            if (j == 0) P.log_pi[e * n_a + ag] = lp;
        }
    }
}


// =====================================================================================================
// Tensor-core path: the same network as ONE persistent tcgen05 kernel (5th-generation tensor cores, accumulators and
// the activation operand in tensor memory).
//
//   * one CTA per SM; warps 0-3 ("compute"): thread t owns TMEM lane t = one agent ("column") of the current 128-agent
//     tile; warps 4-7 ("loader") convert the NEXT tile's observations into the second operand-A buffer meanwhile;
//   * the three 192x192 weight matrices live in shared memory for the whole kernel as fp16 in the canonical K-major
//     no-swizzle UMMA layout (8-row x 16-byte core matrices; prepared on the host, pulled in by three bulk async copies):
//     3 x 73 728 B — which is why this path is fp16: fp32/tf32 weights would not fit next to each other;
//   * activations never touch shared or global memory: obs -> registers -> fp16 -> tcgen05.st -> TMEM (operand A);
//     tcgen05.mma (M128 N192 K16, twelve per layer, issued by one thread) accumulates fp32 in TMEM; after
//     tcgen05.commit -> mbarrier every thread pulls its row back with tcgen05.ld, adds the bias, applies leaky_relu and
//     stores the fp16 result over operand A for the next layer;
//   * the 180 -> 2 output layer, tanh, exploration noise and log-prob run on the fp32 registers of the last epilogue.
// Arithmetic: fp16 operands (11-bit significands), fp32 accumulation: deviates from the fp32 network by ~1e-3 absolute on
// the tanh output ("fast mode"; the exact path is k_policy_mlp above).
// =====================================================================================================
constexpr int TC_M = 128;                                   // agents per tile = TMEM lanes
constexpr int TC_N = POL_HP;                                // 192 outputs per layer
constexpr int TC_W_BYTES = POL_HP * POL_HP * 2;             // one layer of fp16 weights, canonical layout
constexpr int TC_LBO = (POL_HP / 8) * 128;                  // bytes between the two 16-byte k-chunks of one MMA (next core-matrix column)
constexpr int TC_SBO = 128;                                 // bytes between 8-row groups
constexpr int TC_COL_D = 0, TC_COL_A = 256, TC_COLS = 512;  // TMEM columns: accumulator [0,192), operand A [256,352)
// instruction descriptor (cute::UMMA::InstrDescriptor): D fp32, A/B fp16, both K-major, N = 192, M = 128
constexpr uint32_t TC_IDESC = (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(TC_N >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
constexpr int TC_AMAX = 4;                                  // largest action dimension of the tensor-core path (shared-memory budget)
__host__ __device__ constexpr size_t tc_smem_bytes(int A) {  // weights + biases + output layer + partial outputs + barriers
    return (size_t)3 * TC_W_BYTES + 3 * POL_HP * 4 + (size_t)A * POL_HP * 4 + (size_t)((A + 1) & ~1) * 4 + (size_t)TC_M * A * 4 + 96;
}

__device__ __forceinline__ uint32_t s_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(s_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor), K-major, SWIZZLE_NONE, version 1 (Blackwell)
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)((TC_LBO >> 4) & 0x3fff) << 16) | ((uint64_t)((TC_SBO >> 4) & 0x3fff) << 32) |
           (1ull << 46);
}
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);            // .x = lo -> bits [0,16): the lower k index sits in the lower half
    return *reinterpret_cast<const uint32_t *>(&h);
}

#define TC_LD32(taddr, v)                                                                                              \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];" \
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),   \
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),      \
                   "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),     \
                   "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])                                                                       \
                 : "r"(taddr) : "memory")
#define TC_ST16(taddr, v)                                                                                              \
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"                   \
                 :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), \
                    "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory")

struct PolicyTcParams {
    PolicyParams base;                 // obs / act / log_pi / sizes / exploration (weight pointers unused)
    const unsigned char *w16;          // [3][TC_W_BYTES] fp16 weights in canonical UMMA layout (device)
    const float *small;                // b[3][192], W4[A][192], b4[A] fp32 (device)
    float *debug;                      // optional [n_cols][192] fp32: layer-1 pre-activations (tests), or NULL
    long n_tiles;
};

constexpr int TC_LOADERS = 2;               // loader warps per TMEM lane quadrant (each converts 192 / TC_LOADERS features of a row)
constexpr int TC_EPI = 2;                   // epilogue warps per TMEM lane quadrant (each handles 192 / TC_EPI accumulator columns of a row)
constexpr int TC_CTHREADS = TC_EPI * TC_M;  // warps 0-7: MMA issue (thread 0) + epilogues ("compute")
constexpr int TC_THREADS = (TC_EPI + TC_LOADERS) * TC_M;   // warps 8-15: observation loaders
constexpr int TC_COL_A1 = TC_COL_A + POL_HP / 2;   // second operand-A buffer (the loader fills one while the other is in use)

__device__ __forceinline__ void tc_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void tc_mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t *bar) {      // arrives on bar once every tcgen05.mma issued so far has retired
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s_u32(bar)) : "memory");
}

__device__ __forceinline__ void tc_expect_tx(uint64_t *bar, uint32_t bytes) {  // bar also waits for `bytes` of bulk copies
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_bulk_load(void *smem, const void *gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(s_u32(smem)), "l"(gmem), "r"(bytes), "r"(s_u32(bar)) : "memory");
}

// ---- pieces shared by the two tcgen05 kernels
// biases and output layer -> shared memory: the kernels carve sB [3][192], sW4 [A][192] and sb4 [A] back to back, the same
// order as Q.small, so this is one copy of 3 * 192 + A * 192 + A floats
__device__ __forceinline__ void tc_load_small(const float *small, float *sB, int A, int tid, int nthreads) {
    for (int k = tid; k < 3 * POL_HP + A * POL_HP + A; k += nthreads) sB[k] = small[k];
}

// one warp allocates the tensor memory of this SM; the barrier also publishes everything the CTA set up before the call
__device__ __forceinline__ uint32_t tc_tmem_alloc(uint32_t *tmem_slot, int warp) {
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_u32(tmem_slot)), "r"((uint32_t)TC_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    return *tmem_slot;
}
__device__ __forceinline__ void tc_tmem_free(uint32_t tmem, int warp) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)TC_COLS) : "memory");
}

// pull the observations of tile nt (a contiguous run of whole envs) into the L2 while the current tile is converted
__device__ __forceinline__ void tc_prefetch_tile(const PolicyParams &P, long nt, long n_tiles) {
    if (nt >= n_tiles) return;
    const int n_a = P.n_a;
    const long e0 = nt * TC_M / n_a;
    long e1 = (nt * TC_M + TC_M - 1) / n_a; if (e1 * n_a >= P.n_cols) e1 = (P.n_cols - 1) / n_a;
    const size_t env_bytes = (size_t)P.K0 * n_a * sizeof(float);
    if ((env_bytes & 15) == 0)
        for (long ee = e0; ee <= e1; ++ee)
            for (size_t off = 0; off < env_bytes; off += 32768) {
                const uint32_t sz = (uint32_t)(env_bytes - off < 32768 ? env_bytes - off : 32768);
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<const char *>(P.obs) + ee * env_bytes + off), "r"(sz) : "memory");
            }
}

// loader: features k0..k0+31 of column col = agent ag of env e (zero beyond K0 and for dead columns) -> f.  ROWS: also
// store them as the chunk of the column's replay row (swarm_policy_rows_out).
template <bool ROWS>
__device__ __forceinline__ void tc_load_obs32(const PolicyParams &P, long col, bool valid, long e, int ag, int k0, float (&f)[32]) {
    if (P.obs_am && (P.K0 & 3) == 0 && k0 + 32 <= P.K0) {
        // agent-major observations: this thread's 32 features are 128 contiguous bytes of the agent's row
        const float4 *r4 = reinterpret_cast<const float4 *>(P.obs + col * (long)P.K0 + k0);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 v = valid ? __ldg(r4 + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            f[4 * q] = v.x; f[4 * q + 1] = v.y; f[4 * q + 2] = v.z; f[4 * q + 3] = v.w;
        }
    } else if (P.obs_am) {
#pragma unroll
        for (int q = 0; q < 32; ++q) {
            const int k = k0 + q;
            f[q] = (valid && k < P.K0) ? __ldg(P.obs + col * (long)P.K0 + k) : 0.f;
        }
    } else {
#pragma unroll
        for (int q = 0; q < 32; ++q) {
            const int k = k0 + q;
            f[q] = (valid && k < P.K0) ? __ldg(P.obs + (e * P.K0 + k) * P.n_a + ag) : 0.f;
        }
    }
    if (ROWS && valid) {                                    // the row chunk this thread holds: 128 contiguous bytes
        float *rw = P.rows_out + col * P.K0 + k0;
        if ((P.K0 & 3) == 0 && k0 + 32 <= P.K0) {
#pragma unroll
            for (int q = 0; q < 8; ++q) reinterpret_cast<float4 *>(rw)[q] = make_float4(f[4 * q], f[4 * q + 1], f[4 * q + 2], f[4 * q + 3]);
        } else {
#pragma unroll
            for (int q = 0; q < 32; ++q) if (k0 + q < P.K0) rw[q] = f[q];
        }
    }
}

// MMA thread: D (+)= A W^T over K = 192, twelve tcgen05.mma of K = 16 (two 16-byte k-chunks each); accumulate = false
// makes the first one overwrite D
__device__ __forceinline__ void tc_mma_k192(uint32_t d_tmem, uint32_t a_tmem, uint32_t wbase, bool accumulate) {
#pragma unroll 1
    for (int j = 0; j < POL_HP / 16; ++j) {
        const uint64_t bdesc = tc_smem_desc(wbase + (uint32_t)j * 2u * TC_LBO);
        const uint32_t acc = (accumulate || j > 0) ? 1u : 0u;
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
            ::"r"(d_tmem), "r"(a_tmem + j * 8), "l"(bdesc), "r"(TC_IDESC), "r"(acc), "r"(0u) : "memory");
    }
}

// epilogue: 32 accumulator columns of this thread's row -> h = leaky_relu(acc + bias); dbg (or NULL) receives the raw
// accumulators
__device__ __forceinline__ void tc_bias_act32(uint32_t taddr, const float *bias, float slope, float *dbg, float (&h)[32]) {
    uint32_t v[32];
    TC_LD32(taddr, v);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    if (dbg) {
#pragma unroll
        for (int q = 0; q < 32; ++q) dbg[q] = __uint_as_float(v[q]);
    }
#pragma unroll
    for (int q4 = 0; q4 < 8; ++q4) {
        const float4 b4v = *reinterpret_cast<const float4 *>(bias + q4 * 4);
        const float bb[4] = {b4v.x, b4v.y, b4v.z, b4v.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float s_ = __uint_as_float(v[q4 * 4 + u]) + bb[u];
            h[q4 * 4 + u] = s_ > 0.f ? s_ : s_ * slope;
        }
    }
}

// last layer's epilogue: out[j] += the 32 h3 values times the matching output-layer weights w4 = sW4 + 32 c
__device__ __forceinline__ void tc_out_acc32(const float (&h)[32], const float *w4, int A, float (&out)[TC_AMAX]) {
#pragma unroll
    for (int j = 0; j < TC_AMAX; ++j) {
        if (j < A) {
            float s_ = out[j];
#pragma unroll
            for (int q4 = 0; q4 < 8; ++q4) {
                const float4 w = *reinterpret_cast<const float4 *>(w4 + j * POL_HP + q4 * 4);
                s_ = fmaf(h[q4 * 4], w.x, s_); s_ = fmaf(h[q4 * 4 + 1], w.y, s_);
                s_ = fmaf(h[q4 * 4 + 2], w.z, s_); s_ = fmaf(h[q4 * 4 + 3], w.w, s_);
            }
            out[j] = s_;
        }
    }
}

// end of a tile: the second column half hands its partial outputs to the first, which finishes the row with tanh,
// exploration and the act / log_pi stores (same definitions as k_policy_mlp).  The barrier also orders every compute
// thread's accumulator reads before thread 0 starts the next tile's first MMA.
__device__ __forceinline__ void tc_finish_row(const PolicyParams &P, const float (&out)[TC_AMAX], float *s_part, const float *sb4,
                                              int row, int half, long col, bool valid) {
    const int A = P.A, n_a = P.n_a;
    if (half == 1) {
#pragma unroll
        for (int j = 0; j < TC_AMAX; ++j) if (j < A) s_part[row * A + j] = out[j];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("bar.sync 1, %0;" ::"n"(TC_CTHREADS) : "memory");
    if (!valid || half != 0) return;
    const long e = col / n_a; const int ag = (int)(col - e * n_a);
    float q2 = 0.f;
#pragma unroll
    for (int j = 0; j < TC_AMAX; ++j) {
        if (j >= A) break;
        float a = tanhf((out[j] + s_part[row * A + j]) + sb4[j]);
        if (P.explore == 1) {
            const float g = pol_gauss(P, col, j);
            q2 += g * g;
            a = fminf(fmaxf(a + g * P.scale, -1.f), 1.f);
        } else if (P.explore == 2) {
            a = pol_uniform(P, col, j);
        }
        P.act[(e * A + j) * n_a + ag] = a;
    }
    if (P.log_pi) {
        float lp = 0.f;
        if (P.explore == 2) lp = -(float)A * 0.69314718056f;
        else if (P.explore == 1) lp = -0.5f * q2 - (float)A * logf(P.scale * 2.50662827463f);
        P.log_pi[e * n_a + ag] = lp;
    }
}

template <bool ROWS>   // ROWS: the loaders also write every agent's observation as a replay row (swarm_policy_rows_out)
__global__ void __launch_bounds__(TC_THREADS, 1) k_policy_mlp_tc(const PolicyTcParams Q) {
    extern __shared__ __align__(128) unsigned char tsm[];
    unsigned char *sW = tsm;                                             // 3 layers of weights
    float *sB = reinterpret_cast<float *>(sW + 3 * TC_W_BYTES);          // [3][192]
    float *sW4 = sB + 3 * POL_HP;                                        // [A][192]
    float *sb4 = sW4 + Q.base.A * POL_HP;                                // [A], padded to an even count
    float *s_part = sb4 + ((Q.base.A + 1) & ~1);                         // [TC_M][A] partial outputs of the second column half
    uint64_t *bar_w = reinterpret_cast<uint64_t *>(s_part + TC_M * Q.base.A);   // weights landed
    uint64_t *bar_mma = bar_w + 1;                                       // a layer's MMAs retired
    uint64_t *bar_full = bar_mma + 1;                                    // [2] loader -> compute: operand-A buffer b holds a tile's observations
    uint64_t *bar_free = bar_full + 2;                                   // [2] compute -> loader: the last MMA reading buffer b has retired
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bar_free + 2);
    const PolicyParams &P = Q.base;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int n_a = P.n_a;

    if (tid == 0) {
        tc_mbar_init(bar_w, 1); tc_mbar_init(bar_mma, 1);
        tc_mbar_init(&bar_full[0], TC_LOADERS * TC_M); tc_mbar_init(&bar_full[1], TC_LOADERS * TC_M);
        tc_mbar_init(&bar_free[0], 1); tc_mbar_init(&bar_free[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        tc_expect_tx(bar_w, 3u * TC_W_BYTES);
        for (int l = 0; l < 3; ++l) tc_bulk_load(sW + l * TC_W_BYTES, Q.w16 + (size_t)l * TC_W_BYTES, (uint32_t)TC_W_BYTES, bar_w);
    }
    tc_load_small(Q.small, sB, P.A, tid, TC_THREADS);
    const uint32_t tmem = tc_tmem_alloc(tmem_slot, warp);
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);   // a warp reaches the TMEM lane quadrant warp % 4
    const int row = tid & (TC_M - 1);                                    // TMEM lane = agent of the tile

    if (warp >= 4 * TC_EPI) {
        // ================= loader: observation row -> fp16 -> operand-A buffer (it & 1), one tile ahead of the MMAs
        int it = 0;
#pragma unroll 1
        for (long tile = blockIdx.x; tile < Q.n_tiles; tile += gridDim.x, ++it) {
            const int b = it & 1;
            if (tid == TC_CTHREADS) tc_prefetch_tile(P, tile + gridDim.x, Q.n_tiles);
            if (it >= 2) tc_mbar_wait(&bar_free[b], (uint32_t)((it >> 1) - 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const long col = tile * TC_M + row;
            const bool valid = col < P.n_cols;
            const long e = valid ? col / n_a : 0; const int ag = valid ? (int)(col - e * n_a) : 0;
            const uint32_t abase = lane_base + (b ? TC_COL_A1 : TC_COL_A);
            constexpr int FPL = POL_HP / TC_LOADERS;                     // features per loader thread
            const int k_lo = ((warp - 4 * TC_EPI) >> 2) * FPL;
#pragma unroll 1
            for (int c = 0; c < FPL / 32; ++c) {                         // 32 loads in flight per thread and batch (register budget: 512 threads)
                float f[32];
                tc_load_obs32<ROWS>(P, col, valid, e, ag, k_lo + c * 32, f);
                uint32_t r[16];
#pragma unroll
                for (int q = 0; q < 16; ++q) r[q] = pack_h2(f[2 * q], f[2 * q + 1]);
                TC_ST16(abase + (k_lo >> 1) + c * 16, r);
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            tc_mbar_arrive(&bar_full[b]);
        }
    } else {
        // ================= compute: thread 0 issues the MMAs; two warps per lane quadrant share a row's epilogue (96 columns each)
        const int half = warp >> 2;
        uint32_t par_mma = 0;
        int it = 0;
#pragma unroll 1
        for (long tile = blockIdx.x; tile < Q.n_tiles; tile += gridDim.x, ++it) {
            const int b = it & 1;
            const uint32_t acol = b ? TC_COL_A1 : TC_COL_A;
            const long col = tile * TC_M + row;
            const bool valid = col < P.n_cols;
            float *dbg = Q.debug && valid ? Q.debug + col * POL_HP : nullptr;
            float out[TC_AMAX];
#pragma unroll
            for (int j = 0; j < TC_AMAX; ++j) out[j] = 0.f;
#pragma unroll 1
            for (int layer = 0; layer < 3; ++layer) {
                if (layer > 0) {                                         // operand A rewritten by every epilogue thread
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    asm volatile("bar.sync 1, %0;" ::"n"(TC_CTHREADS) : "memory");
                }
                if (tid == 0) {
                    if (it == 0 && layer == 0) tc_mbar_wait(bar_w, 0);
                    if (layer == 0) tc_mbar_wait(&bar_full[b], (uint32_t)(it >> 1) & 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    tc_mma_k192(tmem + TC_COL_D, tmem + acol, s_u32(sW + layer * TC_W_BYTES), false);
                    tc_commit(bar_mma);
                    if (layer == 2) tc_commit(&bar_free[b]);             // buffer b may be refilled once these MMAs have retired
                }
                tc_mbar_wait(bar_mma, par_mma); par_mma ^= 1u;
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
                for (int c = half * (POL_HP / 32 / TC_EPI); c < (half + 1) * (POL_HP / 32 / TC_EPI); ++c) {   // 32 accumulator columns at a time
                    float h[32];
                    tc_bias_act32(lane_base + TC_COL_D + c * 32, sB + layer * POL_HP + c * 32, P.slope, layer == 0 && dbg ? dbg + c * 32 : nullptr, h);
                    if (layer < 2) {
                        uint32_t r[16];
#pragma unroll
                        for (int q = 0; q < 16; ++q) r[q] = pack_h2(h[2 * q], h[2 * q + 1]);
                        TC_ST16(lane_base + acol + c * 16, r);
                    } else {
                        tc_out_acc32(h, sW4 + c * 32, P.A, out);
                    }
                }
                if (layer < 2) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            }
            tc_finish_row(P, out, s_part, sb4, row, half, col, valid);
        }
    }
    tc_tmem_free(tmem, warp);
}

// =====================================================================================================
// fp32-accurate tensor-core path: every fp32 operand x is split into two fp16 numbers, hi = fp16(x) and lo = fp16(x - hi)
// (22 significant bits together; fp16 x fp16 products are exact in the fp32 accumulator), and each layer runs
//     D  =  A_hi W_hi^T  +  A_lo W_hi^T  +  A_hi W_lo^T          (the lo x lo term, 2^-22 relative, is dropped)
// as 3 x 12 tcgen05.mma into ONE fp32 accumulator.  Weights are now 2 x 73 728 B per layer, so they cannot all stay
// resident: a dedicated producer warp streams the six chunks H1 L1 H2 L2 H3 L3 (L2-resident) round and round through a
// 3-slot shared-memory ring with bulk async copies; full[slot] (expect_tx) tells the MMA thread a chunk has landed,
// free[slot] (tcgen05.commit after the last MMA reading it) tells the producer it may be overwritten.
// TMEM: accumulator [0,192), A_hi [192,288), A_lo [288,384) — no room for a second operand buffer, so the loaders
// refill the operand only after the tile's last MMA has retired (the next tile's observations are prefetched into the L2).
// Values beyond the fp16 range (|x| > 65504) saturate.
// =====================================================================================================
constexpr int T3_COL_AH = 192, T3_COL_AL = 288;
constexpr int T3_THREADS = TC_THREADS + 32;     // + the weight-streaming warp

__device__ __forceinline__ void split_h2(float a, float b, uint32_t &hi, uint32_t &lo) {
    a = fminf(fmaxf(a, -65504.f), 65504.f); b = fminf(fmaxf(b, -65504.f), 65504.f);
    const __half2 h = __floats2half2_rn(a, b);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);            // exact differences
    hi = *reinterpret_cast<const uint32_t *>(&h); lo = *reinterpret_cast<const uint32_t *>(&l);
}

template <bool ROWS>
__global__ void __launch_bounds__(T3_THREADS, 1) k_policy_mlp_tc3(const PolicyTcParams Q) {
    extern __shared__ __align__(128) unsigned char tsm[];
    unsigned char *sW = tsm;                                             // 3 ring slots of TC_W_BYTES
    float *sB = reinterpret_cast<float *>(sW + 3 * TC_W_BYTES);          // [3][192]
    float *sW4 = sB + 3 * POL_HP;                                        // [A][192]
    float *sb4 = sW4 + Q.base.A * POL_HP;                                // [A], padded to an even count
    float *s_part = sb4 + ((Q.base.A + 1) & ~1);                         // [TC_M][A] partial outputs of the second column half
    uint64_t *bar_mma = reinterpret_cast<uint64_t *>(s_part + TC_M * Q.base.A);   // a layer's MMAs retired
    uint64_t *bar_afull = bar_mma + 1;                                   // loaders -> MMA thread: operand holds the tile's observations
    uint64_t *bar_afree = bar_afull + 1;                                 // MMA thread -> loaders: the tile's last MMA retired
    uint64_t *bar_full = bar_afree + 1;                                  // [3] weight chunk landed in slot
    uint64_t *bar_free = bar_full + 3;                                   // [3] last MMA reading the slot retired
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bar_free + 3);
    const PolicyParams &P = Q.base;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int n_a = P.n_a;
    const long my_tiles = (Q.n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;

    if (tid == 0) {
        tc_mbar_init(bar_mma, 1); tc_mbar_init(bar_afull, TC_LOADERS * TC_M); tc_mbar_init(bar_afree, 1);
        for (int k = 0; k < 3; ++k) { tc_mbar_init(&bar_full[k], 1); tc_mbar_init(&bar_free[k], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_load_small(Q.small, sB, P.A, tid, T3_THREADS);
    const uint32_t tmem = tc_tmem_alloc(tmem_slot, warp);
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int row = tid & (TC_M - 1);

    if (warp == 4 * (TC_EPI + TC_LOADERS)) {
        // ================= weight producer (one lane): chunk k of the endless sequence H1 L1 H2 L2 H3 L3 ... -> slot k % 3
        if ((tid & 31) == 0) {
            const long n_chunks = 6 * my_tiles;
#pragma unroll 1
            for (long k = 0; k < n_chunks; ++k) {
                const int slot = (int)(k % 3);
                if (k >= 3) tc_mbar_wait(&bar_free[slot], (uint32_t)((k / 3 - 1) & 1));
                tc_expect_tx(&bar_full[slot], (uint32_t)TC_W_BYTES);
                tc_bulk_load(sW + slot * TC_W_BYTES, Q.w16 + (size_t)(k % 6) * TC_W_BYTES, (uint32_t)TC_W_BYTES, &bar_full[slot]);
            }
        }
    } else if (warp >= 4 * TC_EPI) {
        // ================= loaders: observation row -> (hi, lo) fp16 -> operand A, after the previous tile's last MMA retired
        int it = 0;
#pragma unroll 1
        for (long tile = blockIdx.x; tile < Q.n_tiles; tile += gridDim.x, ++it) {
            if (tid == TC_CTHREADS) tc_prefetch_tile(P, tile + gridDim.x, Q.n_tiles);
            if (it >= 1) tc_mbar_wait(bar_afree, (uint32_t)(it - 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const long col = tile * TC_M + row;
            const bool valid = col < P.n_cols;
            const long e = valid ? col / n_a : 0; const int ag = valid ? (int)(col - e * n_a) : 0;
            constexpr int FPL = POL_HP / TC_LOADERS;
            const int k_lo = ((warp - 4 * TC_EPI) >> 2) * FPL;
#pragma unroll 1
            for (int c = 0; c < FPL / 32; ++c) {
                float f[32];
                tc_load_obs32<ROWS>(P, col, valid, e, ag, k_lo + c * 32, f);
                uint32_t rh[16], rl[16];
#pragma unroll
                for (int q = 0; q < 16; ++q) split_h2(f[2 * q], f[2 * q + 1], rh[q], rl[q]);
                TC_ST16(lane_base + T3_COL_AH + (k_lo >> 1) + c * 16, rh);
                TC_ST16(lane_base + T3_COL_AL + (k_lo >> 1) + c * 16, rl);
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            tc_mbar_arrive(bar_afull);
        }
    } else {
        // ================= compute: thread 0 issues the MMAs; two warps per lane quadrant share a row's epilogue
        const int half = warp >> 2;
        uint32_t par_mma = 0;
        long kc = 0;                                                     // weight-chunk counter (thread 0)
        int it = 0;
#pragma unroll 1
        for (long tile = blockIdx.x; tile < Q.n_tiles; tile += gridDim.x, ++it) {
            const long col = tile * TC_M + row;
            const bool valid = col < P.n_cols;
            float *dbg = Q.debug && valid ? Q.debug + col * POL_HP : nullptr;
            float out[TC_AMAX];
#pragma unroll
            for (int j = 0; j < TC_AMAX; ++j) out[j] = 0.f;
#pragma unroll 1
            for (int layer = 0; layer < 3; ++layer) {
                if (layer > 0) {
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    asm volatile("bar.sync 1, %0;" ::"n"(TC_CTHREADS) : "memory");
                }
                if (tid == 0) {
                    if (layer == 0) tc_mbar_wait(bar_afull, (uint32_t)it & 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
                    for (int g = 0; g < 3; ++g) {                        // (A_hi, H), (A_lo, H), (A_hi, L)
                        const long kk = kc + (g == 2 ? 1 : 0);
                        const int slot = (int)(kk % 3);
                        if (g != 1) { tc_mbar_wait(&bar_full[slot], (uint32_t)((kk / 3) & 1)); asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
                        tc_mma_k192(tmem + TC_COL_D, tmem + (g == 1 ? T3_COL_AL : T3_COL_AH), s_u32(sW + slot * TC_W_BYTES), g > 0);
                        if (g >= 1) tc_commit(&bar_free[slot]);          // H after its second use, L after its only use
                    }
                    kc += 2;
                    tc_commit(bar_mma);
                    if (layer == 2) tc_commit(bar_afree);
                }
                tc_mbar_wait(bar_mma, par_mma); par_mma ^= 1u;
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
                for (int c = half * (POL_HP / 32 / TC_EPI); c < (half + 1) * (POL_HP / 32 / TC_EPI); ++c) {
                    float h[32];
                    tc_bias_act32(lane_base + TC_COL_D + c * 32, sB + layer * POL_HP + c * 32, P.slope, layer == 0 && dbg ? dbg + c * 32 : nullptr, h);
                    if (layer < 2) {
                        uint32_t rh[16], rl[16];
#pragma unroll
                        for (int q = 0; q < 16; ++q) split_h2(h[2 * q], h[2 * q + 1], rh[q], rl[q]);
                        TC_ST16(lane_base + T3_COL_AH + c * 16, rh);
                        TC_ST16(lane_base + T3_COL_AL + c * 16, rl);
                    } else {
                        tc_out_acc32(h, sW4 + c * 32, P.A, out);
                    }
                }
                if (layer < 2) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            }
            tc_finish_row(P, out, s_part, sb4, row, half, col, valid);
        }
    }
    tc_tmem_free(tmem, warp);
}

}  // namespace swarm
