// state_kernels.cuh — sm_100a copy kernel of the state store (swarm_state_save / swarm_state_load, include/swarm_b200.h).
//
// A slot holds one env's complete state: a fixed list of segments, each the env's row of one of the handle's [E][...] arrays,
// at 16-byte aligned offsets of the slot (the layout is built on the host, DESIGN.md §11).  k_state_copy<SAVE> copies those rows
// for a list of (env, slot) pairs: env rows -> slots (SAVE) or slots -> env rows (load).  It is a pure HBM copy.
//
// Work split: CTA (x, y) copies bytes [x * chunk, (x + 1) * chunk) of the slot of pair y, i.e. the parts of every segment that
// fall into that range.  The host picks `chunk` (a multiple of 16) so that even one pair is spread over more CTAs than the machine
// has SMs.  Each (segment, pair) piece is copied with the widest access both addresses allow: slot offsets are 16-byte aligned, env
// rows are not always (in_flags is 4 n_a bytes per env, n_g 4 bytes), so the width is chosen per piece, not per launch.
// A launch never reads and writes the same memory: a save reads env rows and writes slots (distinct), a load reads slots and
// writes the rows of distinct envs.
#pragma once
#include <cuda_runtime.h>

#include <stdint.h>

namespace swarm {

constexpr int STATE_THREADS = 256;
constexpr int STATE_PAIRS_PER_LAUNCH = 2048;          // (env, slot) pairs carried in the kernel parameters (16 KB)
constexpr int STATE_MAX_SEGS = 20;
constexpr int STATE_UNMATCHED = (int)0x80000000u;     // pair.y flag of a load: write shape id -1 (the slot's library differs)

struct StateSeg {
    unsigned char *env;    // row of env e at env + e * row
    long long row;         // bytes per env row (a multiple of 4)
    long long off;         // offset in the slot (a multiple of 16)
    int shape_id;          // this segment is the env's library shape id (d_shape_id)
    int pad_;
};

struct StateCopyParams {
    unsigned char *slots;
    long long slot_bytes;  // a multiple of 128
    long long chunk;       // bytes of a slot per CTA, a multiple of 16
    int n_segs, pad_;
    StateSeg seg[STATE_MAX_SEGS];
    int2 pair[STATE_PAIRS_PER_LAUNCH];   // (env, slot | STATE_UNMATCHED)
};

// n bytes (a multiple of sizeof(T)) from src to dst by the whole CTA, four accesses in flight per thread
template <typename T>
__device__ __forceinline__ void state_copy_words(unsigned char *__restrict__ dst, const unsigned char *__restrict__ src, long long n) {
    T *d = reinterpret_cast<T *>(dst);
    const T *s = reinterpret_cast<const T *>(src);
    const long long m = n / (long long)sizeof(T);
    long long i = threadIdx.x;
    for (; i + 3 * STATE_THREADS < m; i += 4 * STATE_THREADS) {
        const T a = s[i], b = s[i + STATE_THREADS], c = s[i + 2 * STATE_THREADS], e = s[i + 3 * STATE_THREADS];
        d[i] = a; d[i + STATE_THREADS] = b; d[i + 2 * STATE_THREADS] = c; d[i + 3 * STATE_THREADS] = e;
    }
    for (; i < m; i += STATE_THREADS) d[i] = s[i];
}

template <bool SAVE>
__global__ void __launch_bounds__(STATE_THREADS) k_state_copy(const __grid_constant__ StateCopyParams P) {
    const int2 pr = P.pair[blockIdx.y];
    const long long e = pr.x, slot = pr.y & 0x7FFFFFFF;
    const long long c0 = (long long)blockIdx.x * P.chunk, c1 = c0 + P.chunk;
    unsigned char *const slot_base = P.slots + slot * P.slot_bytes;
    for (int g = 0; g < P.n_segs; ++g) {
        const StateSeg S = P.seg[g];
        const long long lo = max(c0, S.off), hi = min(c1, S.off + S.row);
        if (lo >= hi) continue;
        unsigned char *const ep = S.env + e * S.row + (lo - S.off);
        unsigned char *const sp = slot_base + lo;
        if (!SAVE && S.shape_id && (pr.y & STATE_UNMATCHED)) {          // restored as unmatched: the general scan serves it
            if (threadIdx.x == 0) *reinterpret_cast<int *>(ep) = -1;
            continue;
        }
        unsigned char *const dst = SAVE ? sp : ep;
        const unsigned char *const src = SAVE ? ep : sp;
        const long long n = hi - lo;
        const unsigned a = (unsigned)(reinterpret_cast<uintptr_t>(ep) | reinterpret_cast<uintptr_t>(sp));
        long long done = 0;
        if ((a & 15) == 0) { done = n & ~15ll; state_copy_words<uint4>(dst, src, done); }
        else if ((a & 7) == 0) { done = n & ~7ll; state_copy_words<uint2>(dst, src, done); }
        state_copy_words<unsigned>(dst + done, src + done, n - done);      // the rest in 4-byte words
    }
}

}  // namespace swarm
