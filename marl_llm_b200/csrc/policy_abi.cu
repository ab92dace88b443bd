// policy_abi.cu — C ABI of the on-device rollout policy (include/swarm_b200.h, group 4).  No CPU implementation.
#include "policy_kernels.cuh"
#include "../../include/swarm_b200.h"

#include <cuda_fp16.h>

#include <string>
#include <vector>

using namespace swarm;

extern "C" int swarm_set_last_error_(int code, const char *msg);   // swarm_abi.cu

namespace {
int pfail(int code, const std::string &m) { return swarm_set_last_error_(code, m.c_str()); }
#define PCU_TRY(expr)                                                                                   \
    do {                                                                                                \
        cudaError_t err__ = (expr);                                                                     \
        if (err__ != cudaSuccess) return pfail(SWARM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(err__)); \
    } while (0)
constexpr size_t POL_SMEM = ((size_t)2 * POL_HP * POL_M + (size_t)2 * POL_KC * POL_HP) * sizeof(float);

// the kernel swarm_policy_step launches for a precision (SWARM_POLICY_*) and rows_out on or off, with its block size and
// its dynamic shared memory for act_dim A (the FFMA kernel writes rows_out without a template switch)
struct PolicyKernel { const void *fn; int threads; size_t smem; };
PolicyKernel policy_kernel(int precision, bool rows, int A) {
    static const void *const fn[3][2] = {
        {(const void *)k_policy_mlp, (const void *)k_policy_mlp},
        {(const void *)k_policy_mlp_tc<false>, (const void *)k_policy_mlp_tc<true>},
        {(const void *)k_policy_mlp_tc3<false>, (const void *)k_policy_mlp_tc3<true>}};
    static const int threads[3] = {POL_THREADS, TC_THREADS, T3_THREADS};
    return {fn[precision][rows], threads[precision], precision == SWARM_POLICY_FP32 ? POL_SMEM : tc_smem_bytes(A)};
}

// byte offset of W[n][k] in one layer of the tensor-core paths' weights: the canonical K-major no-swizzle UMMA layout,
// 8-row x 16-byte core matrices
size_t umma_byte(int k, int n) { return (size_t)(k / 8) * TC_LBO + (size_t)(n / 8) * TC_SBO + (size_t)(n % 8) * 16 + (size_t)(k % 8) * 2; }
}  // namespace

struct swarm_policy {
    int device, obs_dim, hidden, act_dim;
    float *d_w;          // one allocation: Wt[3][HP][HP], b[3][HP], W4[A][HP], b4[A]
    unsigned char *d_w16; // [3][TC_W_BYTES] fp16 weights in the canonical UMMA K-major layout (tensor-core path)
    unsigned char *d_w16x; // [6][TC_W_BYTES] hi/lo fp16 split of the weights, chunk order H1 L1 H2 L2 H3 L3 (fp32-accurate tensor-core path)
    int precision;       // SWARM_POLICY_FP32 | SWARM_POLICY_F16_TC | SWARM_POLICY_F16X3_TC
    int n_sm;
    float *debug;        // test hook: layer-1 accumulators of the tensor-core path
    float *rows_out;     // optional agent-major copy of the observations (swarm_policy_rows_out)
    int obs_am;          // the observations passed to swarm_policy_step are agent-major rows (swarm_policy_obs_layout)
    bool loaded;
    int64_t launches;
};

extern "C" {

int swarm_policy_create(int32_t device, int32_t obs_dim, int32_t hidden_dim, int32_t act_dim, swarm_policy **out) {
    if (!out) return pfail(SWARM_ERR_INVALID, "null argument");
    if (obs_dim <= 0 || obs_dim > POL_HP || hidden_dim <= 0 || hidden_dim > POL_HP || act_dim <= 0 || act_dim > POL_AMAX)
        return pfail(SWARM_ERR_UNSUPPORTED, "policy sizes: obs_dim, hidden_dim <= 192, act_dim <= 8");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return pfail(SWARM_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return pfail(SWARM_ERR_INVALID, "device ordinal out of range");
    PCU_TRY(cudaSetDevice(device));
    swarm_policy *p = new swarm_policy();
    p->device = device; p->obs_dim = obs_dim; p->hidden = hidden_dim; p->act_dim = act_dim; p->loaded = false; p->launches = 0;
    p->precision = SWARM_POLICY_FP32; p->debug = nullptr; p->rows_out = nullptr; p->obs_am = 0; p->d_w16 = nullptr; p->d_w16x = nullptr;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
        delete p;
        return pfail(SWARM_ERR_NO_DEVICE, "device is not sm_100 (kernels are built for sm_100a only)");
    }
    p->n_sm = prop.multiProcessorCount;
    const size_t n = (size_t)3 * POL_HP * POL_HP + 3 * POL_HP + (size_t)act_dim * POL_HP + act_dim;
    cudaError_t e = cudaMalloc(&p->d_w, n * sizeof(float));
    if (e != cudaSuccess) { delete p; return pfail(SWARM_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
    if (e == cudaSuccess) e = cudaMalloc(&p->d_w16, (size_t)3 * TC_W_BYTES);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_w16x, (size_t)6 * TC_W_BYTES);
    for (int prec : {SWARM_POLICY_FP32, SWARM_POLICY_F16_TC, SWARM_POLICY_F16X3_TC})
        for (bool rows : {false, true}) {
            const PolicyKernel k = policy_kernel(prec, rows, TC_AMAX);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem);
        }
    if (e != cudaSuccess) { cudaFree(p->d_w); cudaFree(p->d_w16); cudaFree(p->d_w16x); delete p; return pfail(SWARM_ERR_CUDA, std::string("policy setup: ") + cudaGetErrorString(e)); }
    *out = p;
    return SWARM_OK;
}

int swarm_policy_destroy(swarm_policy *p) {
    if (!p) return SWARM_OK;
    cudaSetDevice(p->device);
    cudaFree(p->d_w);
    cudaFree(p->d_w16);
    cudaFree(p->d_w16x);
    delete p;
    return SWARM_OK;
}

int swarm_policy_load(swarm_policy *p, const float *w1, const float *b1, const float *w2, const float *b2, const float *w3,
                      const float *b3, const float *w4, const float *b4) {
    if (!p || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !w4 || !b4) return pfail(SWARM_ERR_INVALID, "null argument");
    PCU_TRY(cudaSetDevice(p->device));
    const int H = p->hidden, K0 = p->obs_dim, A = p->act_dim;
    const size_t n = (size_t)3 * POL_HP * POL_HP + 3 * POL_HP + (size_t)A * POL_HP + A;
    std::vector<float> h(n, 0.f);
    // every weight W[n][k] (torch Linear.weight is [out][in]) goes to three copies, all zero-padded to 192 x 192:
    //   fp32 path: Wt[k][n];
    //   tensor-core path: fp16 in the UMMA layout (umma_byte);
    //   fp32-accurate tensor-core path: w = hi + lo with hi = fp16(w), lo = fp16(w - hi), same layout, chunks H1 L1 H2 L2 H3 L3
    std::vector<__half> h16((size_t)3 * POL_HP * POL_HP, __float2half(0.f));
    std::vector<__half> hx((size_t)6 * POL_HP * POL_HP, __float2half(0.f));
    const float *W[3] = {w1, w2, w3}, *B[3] = {b1, b2, b3};
    const int Kin[3] = {K0, H, H};
    for (int l = 0; l < 3; ++l) {
        float *wt = h.data() + (size_t)l * POL_HP * POL_HP;
        for (int nn = 0; nn < H; ++nn)
            for (int k = 0; k < Kin[l]; ++k) {
                const float w = W[l][(size_t)nn * Kin[l] + k];
                const size_t u = umma_byte(k, nn) / 2;
                wt[(size_t)k * POL_HP + nn] = w;
                h16[(size_t)l * POL_HP * POL_HP + u] = __float2half_rn(w);
                const float wc = w > 65504.f ? 65504.f : (w < -65504.f ? -65504.f : w);
                const __half hi = __float2half_rn(wc);
                hx[(size_t)(2 * l) * POL_HP * POL_HP + u] = hi;
                hx[(size_t)(2 * l + 1) * POL_HP * POL_HP + u] = __float2half_rn(wc - __half2float(hi));
            }
        float *bb = h.data() + (size_t)3 * POL_HP * POL_HP + (size_t)l * POL_HP;
        for (int nn = 0; nn < H; ++nn) bb[nn] = B[l][nn];
    }
    float *w4p = h.data() + (size_t)3 * POL_HP * POL_HP + 3 * POL_HP;
    for (int j = 0; j < A; ++j)
        for (int k = 0; k < H; ++k) w4p[(size_t)j * POL_HP + k] = w4[(size_t)j * H + k];
    for (int j = 0; j < A; ++j) w4p[(size_t)A * POL_HP + j] = b4[j];
    PCU_TRY(cudaMemcpy(p->d_w, h.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    PCU_TRY(cudaMemcpy(p->d_w16, h16.data(), (size_t)3 * TC_W_BYTES, cudaMemcpyHostToDevice));
    PCU_TRY(cudaMemcpy(p->d_w16x, hx.data(), (size_t)6 * TC_W_BYTES, cudaMemcpyHostToDevice));
    p->loaded = true;
    return SWARM_OK;
}

int swarm_policy_step(swarm_policy *p, const float *obs, int32_t num_envs, int32_t n_a, float *act, float *log_pi, int explore,
                      float noise_scale, uint64_t seed, uint64_t step, void *stream) {
    if (!p || !obs || !act) return pfail(SWARM_ERR_INVALID, "null argument");
    if (!p->loaded) return pfail(SWARM_ERR_INVALID, "swarm_policy_step before swarm_policy_load");
    if (num_envs <= 0 || n_a <= 0 || explore < 0 || explore > 2) return pfail(SWARM_ERR_INVALID, "bad argument");
    PCU_TRY(cudaSetDevice(p->device));
    PolicyParams P;
    P.obs = obs; P.act = act; P.log_pi = log_pi; P.rows_out = p->rows_out; P.obs_am = p->obs_am;
    P.n_cols = (long)num_envs * n_a; P.n_a = n_a; P.K0 = p->obs_dim; P.A = p->act_dim;
    for (int l = 0; l < 3; ++l) {
        P.Wt[l] = p->d_w + (size_t)l * POL_HP * POL_HP;
        P.b[l] = p->d_w + (size_t)3 * POL_HP * POL_HP + (size_t)l * POL_HP;
    }
    P.W4 = p->d_w + (size_t)3 * POL_HP * POL_HP + 3 * POL_HP;
    P.b4 = P.W4 + (size_t)p->act_dim * POL_HP;
    P.slope = 0.01f; P.explore = explore; P.scale = noise_scale; P.seed = seed; P.step = step;
    const PolicyKernel k = policy_kernel(p->precision, p->rows_out != nullptr, p->act_dim);
    PolicyTcParams Q;
    void *args[1] = {&P};
    unsigned grid = (unsigned)((P.n_cols + POL_M - 1) / POL_M);
    if (p->precision != SWARM_POLICY_FP32) {
        Q.base = P; Q.w16 = p->precision == SWARM_POLICY_F16_TC ? p->d_w16 : p->d_w16x;
        Q.small = p->d_w + (size_t)3 * POL_HP * POL_HP; Q.debug = p->debug;
        Q.n_tiles = (P.n_cols + TC_M - 1) / TC_M;
        grid = (unsigned)(Q.n_tiles < p->n_sm ? Q.n_tiles : p->n_sm);     // persistent: one CTA per SM
        args[0] = &Q;
    }
    cudaLaunchKernel(k.fn, dim3(grid), dim3(k.threads), args, k.smem, (cudaStream_t)stream);
    PCU_TRY(cudaGetLastError());                     // returns and clears a launch error, like after a <<<>>> launch
    p->launches++;
    return SWARM_OK;
}

int swarm_policy_set_precision(swarm_policy *p, int precision) {
    if (!p || (precision != SWARM_POLICY_FP32 && precision != SWARM_POLICY_F16_TC && precision != SWARM_POLICY_F16X3_TC))
        return pfail(SWARM_ERR_INVALID, "bad precision");
    if (precision != SWARM_POLICY_FP32 && p->act_dim > TC_AMAX)
        return pfail(SWARM_ERR_UNSUPPORTED, "the tensor-core policy path supports act_dim <= 4 (shared-memory budget)");
    p->precision = precision;
    return SWARM_OK;
}

int swarm_policy_obs_layout(swarm_policy *p, int agent_major) {
    if (!p) return swarm_set_last_error_(SWARM_ERR_INVALID, "null policy");
    p->obs_am = agent_major ? 1 : 0;
    return SWARM_OK;
}

int swarm_policy_rows_out(swarm_policy *p, float *rows_dev) {
    if (!p) return pfail(SWARM_ERR_INVALID, "null handle");
    p->rows_out = rows_dev;
    return SWARM_OK;
}

int swarm_policy_debug_buffer(swarm_policy *p, float *layer1_acc_dev) {
    if (!p) return pfail(SWARM_ERR_INVALID, "null handle");
    p->debug = layer1_acc_dev;
    return SWARM_OK;
}

int64_t swarm_policy_launch_count(const swarm_policy *p) { return p ? p->launches : 0; }

}  // extern "C"
