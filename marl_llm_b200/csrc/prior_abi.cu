// prior_abi.cu — prior policies as programs (include/swarm_b200.h, group 6; DESIGN.md §12): a caller's robot_policy source is
// compiled at run time by NVRTC into an sm_100a CUBIN and loaded as a CUDA library of its own.  This file holds no device code:
// the program's kernels live in the program's CUBIN.  NVRTC is opened with dlopen on the first compile, so the library has no
// link-time dependency on it (or on libcuda: loading goes through the runtime's cudaLibrary* API).
#include "../../include/swarm_b200.h"
#include "../../include/swarm_prior_api.cuh"
#include "prior_program.h"

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

extern "C" int swarm_set_last_error_(int code, const char *msg);   // swarm_abi.cu

namespace {

int qfail(int code, const std::string &m) { return swarm_set_last_error_(code, m.c_str()); }

// include/swarm_prior_api.cuh, embedded at build time (marl_llm_b200/build.py writes swarm_prior_api.inc)
const char kApiHeader[] = {
#include "swarm_prior_api.inc"
    , 0};
const char *const kApiName = "swarm_prior_api.cuh";
// appended to every program: the entry points of the header, after the program's robot_policy
const char *const kEntry = "\n#define SWARM_PRIOR_ENTRY\n#include \"swarm_prior_api.cuh\"\n";
// the library's fixed options: sm_100a, no contraction of products into FMAs, NVRTC's IEEE division and square root
const char *const kOptions[] = {"--gpu-architecture=sm_100a", "--fmad=false", "-default-device"};
const char *const kEntryNames[SWARM_PRIOR_ENTRIES] = {"swarm_prior_f32", "swarm_prior_f64", "swarm_prior_actions"};

// the part of NVRTC's C API the compile uses (nvrtc.h), resolved from the dlopen'ed library
struct Nvrtc {
    void *so = nullptr;
    int (*create)(void **, const char *, const char *, int, const char *const *, const char *const *) = nullptr;
    int (*compile)(void *, int, const char *const *) = nullptr;
    int (*log_size)(void *, size_t *) = nullptr;
    int (*log)(void *, char *) = nullptr;
    int (*cubin_size)(void *, size_t *) = nullptr;
    int (*cubin)(void *, char *) = nullptr;
    int (*destroy)(void **) = nullptr;
};

std::mutex g_mu;                        // guards the two caches below
std::map<std::string, Nvrtc> g_nvrtc;   // by the path asked for
struct LastCompile { std::string source, path, log; std::vector<char> image; bool ok = false; bool valid = false; };
LastCompile g_last;                     // the two-call size query compiles once

int open_nvrtc(const char *path, Nvrtc **out) {
    const std::string want = path ? path : "libnvrtc.so.12";
    const auto it = g_nvrtc.find(want);
    if (it != g_nvrtc.end()) { *out = &it->second; return SWARM_OK; }
    void *so = dlopen(want.c_str(), RTLD_NOW | RTLD_LOCAL);
    if (!so) {
        const char *why = dlerror();
        return qfail(SWARM_ERR_UNSUPPORTED, "NVRTC not found: tried " + want + (why ? std::string(" (") + why + ")" : std::string()) +
                                                (path ? "" : "; pass the path of libnvrtc.so.12 as nvrtc_path"));
    }
    Nvrtc n;
    n.so = so;
    bool ok = true;
    auto sym = [&](auto &fn, const char *name) { void *f = dlsym(so, name); ok = ok && f; fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(f); };
    sym(n.create, "nvrtcCreateProgram"); sym(n.compile, "nvrtcCompileProgram");
    sym(n.log_size, "nvrtcGetProgramLogSize"); sym(n.log, "nvrtcGetProgramLog");
    sym(n.cubin_size, "nvrtcGetCUBINSize"); sym(n.cubin, "nvrtcGetCUBIN"); sym(n.destroy, "nvrtcDestroyProgram");
    if (!ok) {
        dlclose(so);
        return qfail(SWARM_ERR_UNSUPPORTED, "NVRTC not usable: " + want + " lacks the NVRTC entry points (CUBIN output needs CUDA >= 11.1)");
    }
    *out = &(g_nvrtc[want] = n);
    return SWARM_OK;
}

// compiles source into g_last (which keeps the result of the most recent call)
int compile(const char *source, const char *nvrtc_path) {
    const std::string path = nvrtc_path ? nvrtc_path : "";
    if (g_last.valid && g_last.source == source && g_last.path == path) return g_last.ok ? SWARM_OK : SWARM_ERR_INVALID;
    Nvrtc *nv = nullptr;
    if (const int rc = open_nvrtc(nvrtc_path, &nv)) return rc;
    g_last = LastCompile{};
    g_last.source = source; g_last.path = path;
    const std::string full = std::string(source) + kEntry;
    const char *hdr = kApiHeader;
    void *prog = nullptr;
    if (nv->create(&prog, full.c_str(), "robot_policy.cu", 1, &hdr, &kApiName) != 0)
        return qfail(SWARM_ERR_CUDA, "nvrtcCreateProgram failed");
    const int rc = nv->compile(prog, (int)(sizeof(kOptions) / sizeof(kOptions[0])), kOptions);
    size_t n = 0;
    if (nv->log_size(prog, &n) == 0 && n > 1) {
        std::vector<char> log(n);
        if (nv->log(prog, log.data()) == 0) g_last.log.assign(log.data());
    }
    if (rc == 0 && nv->cubin_size(prog, &n) == 0 && n > 0) {
        g_last.image.resize(n);
        g_last.ok = nv->cubin(prog, g_last.image.data()) == 0;
    }
    nv->destroy(&prog);
    g_last.valid = true;
    if (!g_last.ok) return qfail(SWARM_ERR_INVALID, "robot_policy does not compile:\n" + g_last.log);
    return SWARM_OK;
}

}  // namespace

struct swarm_prior_program {
    int device;
    cudaLibrary_t lib;
    cudaKernel_t entry[SWARM_PRIOR_ENTRIES];
};

int swarm_prior_program_device_(const swarm_prior_program *prog) { return prog->device; }

int swarm_prior_program_launch_(const swarm_prior_program *prog, int entry, const swarm_prior_args &args, const int *env_ids,
                                int ctas, int n_a, cudaStream_t stream) {
    const int threads = n_a < 256 ? (n_a + 31) & ~31 : 256;          // k_prior's geometry
    swarm_prior_args a = args;
    a.env_ids = env_ids;
    void *params[] = {&a};
    const cudaError_t e = cudaLaunchKernel((const void *)prog->entry[entry], dim3(ctas), dim3(threads), params, 0, stream);
    if (e != cudaSuccess) return qfail(SWARM_ERR_CUDA, std::string("prior program launch: ") + cudaGetErrorString(e));
    return SWARM_OK;
}

// K programs and an assignment env -> program.  The env ids, grouped by program and ascending within a group, are one device
// array; program k serves the slice [offset[k], offset[k] + count[k]) of it.
struct swarm_prior_population {
    int device, num_envs;
    std::vector<swarm_prior_program *> prog;
    std::vector<int> offset, count;
    int *d_env;
};

int swarm_prior_population_device_(const swarm_prior_population *pop) { return pop->device; }
int swarm_prior_population_envs_(const swarm_prior_population *pop) { return pop->num_envs; }

int swarm_prior_population_launch_(const swarm_prior_population *pop, int entry, const swarm_prior_args &args, int n_a,
                                   cudaStream_t stream, int64_t *launches) {
    for (size_t k = 0; k < pop->prog.size(); ++k) {
        if (pop->count[k] == 0) continue;
        if (const int rc = swarm_prior_program_launch_(pop->prog[k], entry, args, pop->d_env + pop->offset[k], pop->count[k], n_a, stream))
            return rc;
        ++*launches;
    }
    return SWARM_OK;
}

extern "C" {

int swarm_prior_compile(const char *source, const char *nvrtc_path, void *image, int64_t image_cap, int64_t *image_size, char *log,
                        int64_t log_cap) {
    if (!source || !image_size) return qfail(SWARM_ERR_INVALID, "null argument");
    if (image_cap < 0 || log_cap < 0) return qfail(SWARM_ERR_INVALID, "negative capacity");
    std::lock_guard<std::mutex> lock(g_mu);
    const int rc = compile(source, nvrtc_path);
    if (rc == SWARM_ERR_UNSUPPORTED || rc == SWARM_ERR_CUDA) return rc;
    if (log && log_cap > 0) {
        const size_t n = std::min<size_t>(g_last.log.size(), (size_t)log_cap - 1);
        memcpy(log, g_last.log.data(), n);
        log[n] = 0;
    }
    if (rc != SWARM_OK) return qfail(SWARM_ERR_INVALID, "robot_policy does not compile:\n" + g_last.log);
    *image_size = (int64_t)g_last.image.size();
    if (image) {
        if (image_cap < *image_size) return qfail(SWARM_ERR_INVALID, "image_cap is smaller than the image (query the size with image = NULL)");
        memcpy(image, g_last.image.data(), g_last.image.size());
    }
    return SWARM_OK;
}

int swarm_prior_program_create(int32_t device, const void *image, int64_t size, swarm_prior_program **out) {
    if (!image || !out) return qfail(SWARM_ERR_INVALID, "null argument");
    static const unsigned char elf[4] = {0x7f, 'E', 'L', 'F'};
    if (size < 64 || memcmp(image, elf, 4) != 0) return qfail(SWARM_ERR_INVALID, "image is not a CUBIN (swarm_prior_compile's output)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return qfail(SWARM_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return qfail(SWARM_ERR_INVALID, "device ordinal out of range");
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return qfail(SWARM_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    swarm_prior_program *p = new swarm_prior_program();
    p->device = device;
    e = cudaLibraryLoadData(&p->lib, image, nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e != cudaSuccess) {
        delete p;
        return qfail(SWARM_ERR_INVALID, std::string("cudaLibraryLoadData: ") + cudaGetErrorString(e));
    }
    for (int k = 0; k < SWARM_PRIOR_ENTRIES; ++k) {
        e = cudaLibraryGetKernel(&p->entry[k], p->lib, kEntryNames[k]);
        if (e != cudaSuccess) {
            cudaLibraryUnload(p->lib);
            delete p;
            return qfail(SWARM_ERR_INVALID, std::string("the image has no entry point ") + kEntryNames[k]);
        }
    }
    *out = p;
    return SWARM_OK;
}

int swarm_prior_program_destroy(swarm_prior_program *prog) {
    if (!prog) return SWARM_OK;
    cudaSetDevice(prog->device);
    cudaLibraryUnload(prog->lib);
    delete prog;
    return SWARM_OK;
}

int swarm_prior_population_create(int32_t device, int32_t num_envs, int32_t count, swarm_prior_program *const *programs,
                                  const int32_t *env_program, swarm_prior_population **out) {
    if (!programs || !env_program || !out) return qfail(SWARM_ERR_INVALID, "null argument");
    if (count < 1) return qfail(SWARM_ERR_INVALID, "a population needs count >= 1 programs");
    if (num_envs < 1) return qfail(SWARM_ERR_INVALID, "a population needs num_envs >= 1");
    for (int k = 0; k < count; ++k) {
        if (!programs[k]) return qfail(SWARM_ERR_INVALID, "program " + std::to_string(k) + " is NULL");
        if (programs[k]->device != device) return qfail(SWARM_ERR_INVALID, "program " + std::to_string(k) + " is loaded on another device");
    }
    std::vector<int> cnt(count, 0);
    for (int e = 0; e < num_envs; ++e) {
        if (env_program[e] < 0 || env_program[e] >= count)
            return qfail(SWARM_ERR_INVALID, "env_program[" + std::to_string(e) + "] = " + std::to_string(env_program[e]) + " is not in [0, count)");
        cnt[env_program[e]]++;
    }
    std::vector<int> off(count, 0), grouped(num_envs);
    for (int k = 1; k < count; ++k) off[k] = off[k - 1] + cnt[k - 1];
    std::vector<int> fill = off;
    for (int e = 0; e < num_envs; ++e) grouped[fill[env_program[e]]++] = e;
    cudaError_t err = cudaSetDevice(device);
    if (err != cudaSuccess) return qfail(SWARM_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(err));
    int *d_env = nullptr;
    err = cudaMalloc(&d_env, sizeof(int) * (size_t)num_envs);
    if (err == cudaSuccess) err = cudaMemcpy(d_env, grouped.data(), sizeof(int) * (size_t)num_envs, cudaMemcpyHostToDevice);
    if (err != cudaSuccess) {
        if (d_env) cudaFree(d_env);
        return qfail(SWARM_ERR_CUDA, std::string("prior population env list: ") + cudaGetErrorString(err));
    }
    swarm_prior_population *pop = new swarm_prior_population();
    pop->device = device; pop->num_envs = num_envs;
    pop->prog.assign(programs, programs + count);
    pop->offset = off; pop->count = cnt;
    pop->d_env = d_env;
    *out = pop;
    return SWARM_OK;
}

int swarm_prior_population_destroy(swarm_prior_population *pop) {
    if (!pop) return SWARM_OK;
    cudaSetDevice(pop->device);
    cudaFree(pop->d_env);
    delete pop;
    return SWARM_OK;
}

}  // extern "C"
