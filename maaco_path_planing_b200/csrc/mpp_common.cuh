// mpp_common.cuh -- shared device/host helpers for libmpp_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/mpp.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libmpp_b200 is written for sm_100a (B200) only"
#endif

// ---------------------------------------------------------------------------------------------
// error plumbing (never throw across the C ABI)
// ---------------------------------------------------------------------------------------------
void mpp_set_error(const char *fmt, ...);

#define MPP_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            mpp_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return MPP_ECUDA;                                                                   \
        }                                                                                       \
    } while (0)

#define MPP_REQUIRE(cond, ...)          \
    do {                                \
        if (!(cond)) {                  \
            mpp_set_error(__VA_ARGS__); \
            return MPP_EINVAL;          \
        }                               \
    } while (0)

// strategy-1 constants of one map (P1 = orientation start -> target, MAACO.py:146-165)
struct MppS1 {
    uint32_t P1;
    int fast_ok;            // P1 has exactly three moves
    int sm[3];              // those moves
    int dpr[3], dc[3];      // window row pointer delta (bytes) and column delta of each
    int so[3];              // ranking-word offset of (neighbour cell, context move+1)
};
struct MppMapMeta {         // per-map scalars the MAACO kernels read from device memory (one per map of a batch)
    int start, target;
    MppS1 s1;
};
MppMapMeta mpp_make_meta(int rows, int cols, int start, int target);

// A batch of same-shape maps: what every launcher takes (grid.y / blockIdx.y = map); a single map is a batch of one.
struct mpp_map_batch {
    int n_maps, rows, cols, device, sm_count;
    int pitch_words;        // padded occupancy row pitch (32-bit words)
    int occ_words;          // (rows+2)*pitch_words, rounded up to a multiple of 4 words (16 B bulk copies)
    uint32_t *occ_dev;      // [n_maps][occ_words] border-padded bit-packed occupancy; bit (r+1, c+1); border = 1
    uint8_t *svalid_dev;    // [n_maps][rows*cols] static move masks, MAACO move order (bounds/obstacle/corner-cut)
    MppMapMeta *meta_dev;   // [n_maps]
    MppMapMeta *meta_host;  // [n_maps]
    uint8_t *grid_host;     // [n_maps][rows*cols] (host copy for host-side table builds), null for device-built batches
    long long n_obstacles;  // over all maps (0 = no map needs a safety table)
    // safety-class cache of every map (helper.py:67-80); built by mpp_map_batch_safety_table
    double safety_msd;      // msd the tables were built for (<0 = none)
    uint16_t *safety_d2_dev; // [n_maps][rows*cols]: min d^2 to an obstacle inside the (2*floor(msd)+1)^2 stencil, 0 = none
    double *safety_lut_dev; // safety_lut_n doubles, shared by every map (the LUT depends on msd only)
    int safety_lut_n;
};

int mpp_check_device(int device);


// ---------------------------------------------------------------------------------------------
// Philox4x32-10 streams (RNG contract)
// ---------------------------------------------------------------------------------------------
struct mpp_u4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ mpp_u4 mpp_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                        uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
#ifdef __CUDA_ARCH__
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
#else
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t h0 = (uint32_t)(p0 >> 32), l0 = (uint32_t)p0, h1 = (uint32_t)(p1 >> 32), l1 = (uint32_t)p1;
#endif
        uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c0 = n0; c1 = l1; c2 = n2; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    mpp_u4 o = {c0, c1, c2, c3};
    return o;
}

__host__ __device__ __forceinline__ double mpp_u53(uint32_t a, uint32_t b) {
    // exact: (a>>5)*2^26 + (b>>6) < 2^53, then an exact power-of-two scale
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

struct mpp_stream_rng {
    uint32_t k0, k1, cls, it, ind, cursor;
    uint32_t have;  // cached block index + 1 (0 = none)
    mpp_u4 blk;
    __host__ __device__ __forceinline__ void init(uint64_t seed, uint32_t cls_, uint32_t it_, uint32_t ind_) {
        k0 = (uint32_t)seed; k1 = (uint32_t)(seed >> 32); cls = cls_; it = it_; ind = ind_; cursor = 0; have = 0;
    }
    __host__ __device__ __forceinline__ double draw() {
        uint32_t b = cursor >> 1;
        if (have != b + 1) { blk = mpp_philox(b, ind, it, cls, k0, k1); have = b + 1; }
        double u = (cursor & 1) ? mpp_u53(blk.z, blk.w) : mpp_u53(blk.x, blk.y);
        ++cursor;
        return u;
    }
    __host__ __device__ __forceinline__ int below(int n) {  // choice / randint under the tape
        int j = (int)(draw() * (double)n);
        return j < n ? j : n - 1;
    }
};

// ---------------------------------------------------------------------------------------------
// TMA 1-D bulk copy global -> shared with mbarrier completion (SASS: UBLKCP)
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t mpp_smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mpp_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mpp_smem_addr(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mpp_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mpp_smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mpp_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     mpp_smem_addr(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(mpp_smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void mpp_mbar_wait(uint64_t *bar, uint32_t phase) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(mpp_smem_addr(bar)), "r"(phase)
            : "memory");
    }
}
// Stage `bytes` (multiple of 16, 16-B aligned both sides) into shared memory with bulk copies;
// all threads of the block return after the data has landed.
__device__ __forceinline__ void mpp_stage_bulk(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    if (threadIdx.x == 0) {
        mpp_mbar_init(bar, 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mpp_mbar_expect_tx(bar, bytes);
        uint32_t off = 0;
        while (off < bytes) {  // one bulk op moves at most ~1 MB; chunk conservatively
            uint32_t n = bytes - off;
            if (n > 65536u) n = 65536u;
            mpp_bulk_g2s((char *)dst_smem + off, (const char *)src_gmem + off, n, bar);
            off += n;
        }
    }
    mpp_mbar_wait(bar, 0);
}
#endif
