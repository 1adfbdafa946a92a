// mpp_map.cu -- map-batch handle: env.py grids (list-of-lists of 0/1/2/3) -> border-padded,
// bit-packed occupancy tensors in HBM + per-map metadata (the safety-class tables, helper.py:67-80, are in mpp_astar.cu).
#include <stdarg.h>
#include <stdlib.h>

#include <cmath>

#include "mpp_common.cuh"

static thread_local char g_err[512] = "";

void mpp_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" int mpp_abi_version(void) { return MPP_ABI_VERSION; }
extern "C" const char *mpp_last_error(void) { return g_err; }

extern "C" int mpp_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int d = 0; d < n; ++d) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ++ok;
    }
    return ok;
}

int mpp_check_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        mpp_set_error("no CUDA device visible (%s); libmpp_b200 has no CPU fallback",
                      e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return MPP_ENODEVICE;
    }
    if (device < 0 || device >= n) { mpp_set_error("device %d out of range [0,%d)", device, n); return MPP_EINVAL; }
    int major = 0;
    MPP_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) {
        mpp_set_error("device %d is sm_%d0; libmpp_b200 is built for sm_100a only (no fallback)", device, major);
        return MPP_ENODEVICE;
    }
    return MPP_OK;
}

// One thread per padded word: word (pr, pw) holds padded columns [32*pw, 32*pw+32) of padded row pr.
__global__ void mpp_pack_occ_kernel(const uint8_t *__restrict__ grid, int rows, int cols, int pitch_words,
                                    int total_words, uint32_t *__restrict__ occ) {
    int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= total_words) return;
    grid += (size_t)blockIdx.y * rows * cols;                  // blockIdx.y = map of a batch
    occ += (size_t)blockIdx.y * total_words;
    int pr = w / pitch_words, pw = w % pitch_words;
    uint32_t bits = 0;
    if (pr >= rows + 2) { occ[w] = 0xffffffffu; return; }  // tail padding
    int r = pr - 1;
#pragma unroll 4
    for (int b = 0; b < 32; ++b) {
        int c = pw * 32 + b - 1;
        bool blocked = (r < 0 || r >= rows || c < 0 || c >= cols) ? true : (grid[(size_t)r * cols + c] == 1);
        bits |= (blocked ? 1u : 0u) << b;
    }
    occ[w] = bits;
}

// Static per-cell move mask in MAACO's move order (MAACO.py:98): bit m set iff the move stays in bounds,
// lands on a non-obstacle cell (MAACO.py:93-95 without the tabu test) and, for diagonals, does not cut an
// obstacle corner (MAACO.py:100-120).  0 for obstacle cells.
__global__ void mpp_svalid_kernel(const uint32_t *__restrict__ occ, int occ_words, int pitch, int R, int C,
                                  uint8_t *__restrict__ sv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * C) return;
    occ += (size_t)blockIdx.y * occ_words;                     // blockIdx.y = map of a batch
    sv += (size_t)blockIdx.y * R * C;
    const int r = i / C, c = i % C;
    auto blocked = [&](int rr, int cc) -> bool {
        const int pb = cc + 1;
        return (occ[(rr + 1) * pitch + (pb >> 5)] >> (pb & 31)) & 1u;
    };
    uint32_t mask = 0;
    if (!blocked(r, c)) {
        for (int m = 0; m < 8; ++m) {
            const int dr = (int)((0xA940u >> (2 * m)) & 3u) - 1, dc = (int)((0x9224u >> (2 * m)) & 3u) - 1;
            bool ok = !blocked(r + dr, c + dc);
            if (ok && dr != 0 && dc != 0) ok = !blocked(r + dr, c) && !blocked(r, c + dc);
            mask |= (ok ? 1u : 0u) << m;
        }
    }
    sv[i] = (uint8_t)mask;
}

static uint32_t host_orient_mask(int dR, int dC) {                // MAACO.py:146-157
    uint32_t k = 0xffu;
    if (dC > 0) k &= ~0x29u;
    if (dC < 0) k &= ~0x94u;
    if (dR > 0) k &= ~0x07u;
    if (dR < 0) k &= ~0xE0u;
    return k;
}

MppMapMeta mpp_make_meta(int rows, int cols, int start, int target) {
    (void)rows;
    MppMapMeta M;
    memset(&M, 0, sizeof(M));
    M.start = start; M.target = target;
    if (start < 0 || target < 0) return M;
    MppS1 &S = M.s1;
    S.P1 = host_orient_mask(target / cols - start / cols, target % cols - start % cols);
    S.fast_ok = __builtin_popcount(S.P1) == 3;
    uint32_t rest = S.P1;
    for (int i = 0; i < 3; ++i) {
        const int m = S.fast_ok ? __builtin_ctz(rest) : __builtin_ctz(S.P1 ? S.P1 : 1u);
        rest &= rest - 1;
        const int dr = (int)((0xA940u >> (2 * m)) & 3u) - 1, dc = (int)((0x9224u >> (2 * m)) & 3u) - 1;
        S.sm[i] = m; S.dpr[i] = dr * 8; S.dc[i] = dc; S.so[i] = (dr * cols + dc) * 9 + m + 1;
    }
    return M;
}

// A batch of n_maps same-shape maps (BASELINE config 5: independent maps, one launch per colony pass of the
// whole batch; a single map is a batch of one).  grids_host: n_maps * rows * cols bytes.
extern "C" int mpp_map_batch_create(const uint8_t *grids_host, int n_maps, int rows, int cols, int device,
                                    mpp_map_batch **out) {
    MPP_REQUIRE(grids_host && out, "mpp_map_batch_create: null argument");
    MPP_REQUIRE(n_maps > 0 && n_maps <= 65535, "mpp_map_batch_create: n_maps=%d (1..65535)", n_maps);
    MPP_REQUIRE(rows > 0 && cols > 0 && (long long)rows * cols < (1ll << 30), "mpp_map_batch_create: bad shape %dx%d", rows, cols);
    int rc = mpp_check_device(device);
    if (rc) return rc;
    MPP_CUDA(cudaSetDevice(device));
    mpp_map_batch *B = (mpp_map_batch *)calloc(1, sizeof(mpp_map_batch));
    if (!B) { mpp_set_error("out of host memory"); return MPP_ENOMEM; }
    B->n_maps = n_maps; B->rows = rows; B->cols = cols; B->device = device;
    B->safety_msd = -1.0;
    const size_t n = (size_t)rows * cols;
    B->grid_host = (uint8_t *)malloc(n * n_maps);
    B->meta_host = (MppMapMeta *)malloc(sizeof(MppMapMeta) * n_maps);
    if (!B->grid_host || !B->meta_host) { mpp_set_error("out of host memory"); return MPP_ENOMEM; }
    memcpy(B->grid_host, grids_host, n * n_maps);
    for (int k = 0; k < n_maps; ++k) {
        const uint8_t *g = grids_host + n * k;
        int start = -1, target = -1;
        for (size_t i = 0; i < n; ++i) {
            if (g[i] == 2 && start < 0) start = (int)i;             // first row-major hit, MAACO.py:32-41
            if (g[i] == 3 && target < 0) target = (int)i;
            if (g[i] == 1) B->n_obstacles++;
        }
        B->meta_host[k] = mpp_make_meta(rows, cols, start, target);
    }
    B->pitch_words = (cols + 2 + 31) / 32;
    B->occ_words = ((rows + 2) * B->pitch_words + 3) & ~3;
    MPP_CUDA(cudaDeviceGetAttribute(&B->sm_count, cudaDevAttrMultiProcessorCount, device));
    uint8_t *gdev = nullptr;
    MPP_CUDA(cudaMalloc(&gdev, n * n_maps));
    MPP_CUDA(cudaMalloc(&B->occ_dev, (size_t)B->occ_words * 4 * n_maps));
    MPP_CUDA(cudaMalloc(&B->svalid_dev, n * n_maps));
    MPP_CUDA(cudaMalloc(&B->meta_dev, sizeof(MppMapMeta) * n_maps));
    MPP_CUDA(cudaMemcpy(gdev, grids_host, n * n_maps, cudaMemcpyHostToDevice));
    MPP_CUDA(cudaMemcpy(B->meta_dev, B->meta_host, sizeof(MppMapMeta) * n_maps, cudaMemcpyHostToDevice));
    mpp_pack_occ_kernel<<<dim3((B->occ_words + 255) / 256, n_maps), 256>>>(gdev, rows, cols, B->pitch_words, B->occ_words,
                                                                           B->occ_dev);
    MPP_CUDA(cudaGetLastError());
    mpp_svalid_kernel<<<dim3(((int)n + 255) / 256, n_maps), 256>>>(B->occ_dev, B->occ_words, B->pitch_words, rows, cols,
                                                                   B->svalid_dev);
    MPP_CUDA(cudaGetLastError());
    MPP_CUDA(cudaDeviceSynchronize());
    MPP_CUDA(cudaFree(gdev));
    *out = B;
    return MPP_OK;
}

// Device-side ingestion of a batch (mpp_map_batch_create_device), one pass over the cells.  One warp per padded
// occupancy word, lane b = padded column 32*pw + b: a warp reads 32 consecutive cells of one row whatever the element
// width, and the word is a ballot.  Cells are compared raw: clipping to 0..255 (what the host path does) never makes
// or removes a 1, 2 or 3.  A warp walks the words of its map (grid.y = map) in increasing order, so the first start /
// target it meets is its row-major first; per block these fold into ends[map] with atomicMin and the obstacle count
// into *n_obstacles, so the result does not depend on the order blocks run in.  ends must hold MPP_NO_CELL.
#define MPP_NO_CELL 0x7f7f7f7f  // byte pattern 0x7f (cudaMemset); above any cell id (rows*cols < 2^30)
template <typename T>
__global__ void __launch_bounds__(256) mpp_ingest_kernel(const T *__restrict__ grids, int rows, int cols,
                                                         int pitch_words, int total_words, uint32_t *__restrict__ occ,
                                                         int2 *__restrict__ ends,
                                                         unsigned long long *__restrict__ n_obstacles) {
    __shared__ int blk_s, blk_t;
    __shared__ unsigned blk_n;
    const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    if (threadIdx.x == 0) { blk_s = blk_t = MPP_NO_CELL; blk_n = 0; }
    __syncthreads();
    grids += (size_t)blockIdx.y * rows * cols;
    occ += (size_t)blockIdx.y * total_words;
    int first_s = MPP_NO_CELL, first_t = MPP_NO_CELL;
    unsigned n_obs = 0;
    for (int w = blockIdx.x * warps + (threadIdx.x >> 5); w < total_words; w += gridDim.x * warps) {
        const int pr = w / pitch_words, pw = w - pr * pitch_words;
        const int r = pr - 1, c = pw * 32 + lane - 1;
        const bool inside = r >= 0 && r < rows && c >= 0 && c < cols;    // else border or tail padding: blocked
        const T v = inside ? grids[(size_t)r * cols + c] : T(1);
        const uint32_t blocked = __ballot_sync(0xffffffffu, v == T(1));
        const uint32_t s = __ballot_sync(0xffffffffu, inside && v == T(2));
        const uint32_t t = __ballot_sync(0xffffffffu, inside && v == T(3));
        n_obs += __popc(__ballot_sync(0xffffffffu, inside && v == T(1)));
        if (lane == 0) occ[w] = blocked;
        if (s && first_s == MPP_NO_CELL) first_s = r * cols + pw * 32 + __ffs(s) - 2;
        if (t && first_t == MPP_NO_CELL) first_t = r * cols + pw * 32 + __ffs(t) - 2;
    }
    if (lane == 0) {
        if (first_s != MPP_NO_CELL) atomicMin(&blk_s, first_s);
        if (first_t != MPP_NO_CELL) atomicMin(&blk_t, first_t);
        if (n_obs) atomicAdd(&blk_n, n_obs);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (blk_s != MPP_NO_CELL) atomicMin(&ends[blockIdx.y].x, blk_s);
        if (blk_t != MPP_NO_CELL) atomicMin(&ends[blockIdx.y].y, blk_t);
        if (blk_n) atomicAdd(n_obstacles, (unsigned long long)blk_n);
    }
}

static int map_batch_ingest(mpp_map_batch *B, const void *grids_dev, int elem_bytes, cudaStream_t s) {
    const int n_maps = B->n_maps, rows = B->rows, cols = B->cols;
    const size_t n = (size_t)rows * cols;
    B->meta_host = (MppMapMeta *)malloc(sizeof(MppMapMeta) * n_maps);
    if (!B->meta_host) { mpp_set_error("out of host memory"); return MPP_ENOMEM; }
    B->pitch_words = (cols + 2 + 31) / 32;
    B->occ_words = ((rows + 2) * B->pitch_words + 3) & ~3;
    MPP_CUDA(cudaDeviceGetAttribute(&B->sm_count, cudaDevAttrMultiProcessorCount, B->device));
    MPP_CUDA(cudaMalloc(&B->occ_dev, (size_t)B->occ_words * 4 * n_maps));
    MPP_CUDA(cudaMalloc(&B->svalid_dev, n * n_maps));
    MPP_CUDA(cudaMalloc(&B->meta_dev, sizeof(MppMapMeta) * n_maps));
    // what the host reads back -- the obstacle count, then (start, target) per map -- is staged in meta_dev (64 bytes
    // per map) before the metadata built from it overwrites it: no allocation, no cudaFree (a device-wide synchronise)
    static_assert(sizeof(MppMapMeta) >= sizeof(int2) + sizeof(unsigned long long), "scan results must fit meta_dev");
    const size_t scan_bytes = sizeof(unsigned long long) + sizeof(int2) * n_maps;
    unsigned long long *count_dev = (unsigned long long *)B->meta_dev;
    int2 *ends_dev = (int2 *)(count_dev + 1);
    MPP_CUDA(cudaMemsetAsync(count_dev, 0, sizeof(unsigned long long), s));
    MPP_CUDA(cudaMemsetAsync(ends_dev, 0x7f, sizeof(int2) * n_maps, s));
    const int per_map = (B->occ_words + 7) / 8, fill = (B->sm_count * 8 + n_maps - 1) / n_maps;   // ~8 blocks per SM
    const dim3 grid(per_map < fill ? per_map : fill, n_maps);
    if (elem_bytes == 1)
        mpp_ingest_kernel<<<grid, 256, 0, s>>>((const uint8_t *)grids_dev, rows, cols, B->pitch_words, B->occ_words,
                                               B->occ_dev, ends_dev, count_dev);
    else if (elem_bytes == 4)
        mpp_ingest_kernel<<<grid, 256, 0, s>>>((const int32_t *)grids_dev, rows, cols, B->pitch_words, B->occ_words,
                                               B->occ_dev, ends_dev, count_dev);
    else
        mpp_ingest_kernel<<<grid, 256, 0, s>>>((const int64_t *)grids_dev, rows, cols, B->pitch_words, B->occ_words,
                                               B->occ_dev, ends_dev, count_dev);
    MPP_CUDA(cudaGetLastError());
    mpp_svalid_kernel<<<dim3(((int)n + 255) / 256, n_maps), 256, 0, s>>>(B->occ_dev, B->occ_words, B->pitch_words, rows,
                                                                        cols, B->svalid_dev);
    MPP_CUDA(cudaGetLastError());
    unsigned long long *scan = (unsigned long long *)malloc(scan_bytes);
    if (!scan) { mpp_set_error("out of host memory"); return MPP_ENOMEM; }
    cudaError_t e = cudaMemcpyAsync(scan, B->meta_dev, scan_bytes, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
        free(scan);
        MPP_CUDA(e);
    }
    B->n_obstacles = (long long)scan[0];
    const int2 *ends = (const int2 *)(scan + 1);
    for (int k = 0; k < n_maps; ++k) {
        B->meta_host[k] = mpp_make_meta(rows, cols, ends[k].x == MPP_NO_CELL ? -1 : ends[k].x,
                                        ends[k].y == MPP_NO_CELL ? -1 : ends[k].y);
    }
    free(scan);
    MPP_CUDA(cudaMemcpyAsync(B->meta_dev, B->meta_host, sizeof(MppMapMeta) * n_maps, cudaMemcpyHostToDevice, s));
    MPP_CUDA(cudaStreamSynchronize(s));
    return MPP_OK;
}

// A batch from grids already on the device (e.g. written by a torch kernel): nothing crosses to the host but the
// per-map start / target and the obstacle count; grid_host stays null.
extern "C" int mpp_map_batch_create_device(const void *grids_dev, int elem_bytes, int n_maps, int rows, int cols,
                                           int device, void *stream, mpp_map_batch **out) {
    MPP_REQUIRE(grids_dev && out, "mpp_map_batch_create_device: null argument");
    MPP_REQUIRE(elem_bytes == 1 || elem_bytes == 4 || elem_bytes == 8,
                "mpp_map_batch_create_device: elem_bytes=%d (1 = uint8, 4 = int32, 8 = int64)", elem_bytes);
    MPP_REQUIRE(n_maps > 0 && n_maps <= 65535, "mpp_map_batch_create_device: n_maps=%d (1..65535)", n_maps);
    MPP_REQUIRE(rows > 0 && cols > 0 && (long long)rows * cols < (1ll << 30),
                "mpp_map_batch_create_device: bad shape %dx%d", rows, cols);
    int rc = mpp_check_device(device);
    if (rc) return rc;
    MPP_CUDA(cudaSetDevice(device));
    cudaPointerAttributes pa;
    MPP_CUDA(cudaPointerGetAttributes(&pa, grids_dev));
    MPP_REQUIRE((pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged) && pa.device == device,
                "mpp_map_batch_create_device: grids_dev is not memory of device %d", device);
    mpp_map_batch *B = (mpp_map_batch *)calloc(1, sizeof(mpp_map_batch));
    if (!B) { mpp_set_error("out of host memory"); return MPP_ENOMEM; }
    B->n_maps = n_maps; B->rows = rows; B->cols = cols; B->device = device;
    B->safety_msd = -1.0;
    rc = map_batch_ingest(B, grids_dev, elem_bytes, (cudaStream_t)stream);
    if (rc) {
        mpp_map_batch_destroy(B);
        return rc;
    }
    *out = B;
    return MPP_OK;
}

extern "C" void mpp_map_batch_destroy(mpp_map_batch *B) {
    if (!B) return;
    cudaSetDevice(B->device);
    if (B->occ_dev) cudaFree(B->occ_dev);
    if (B->svalid_dev) cudaFree(B->svalid_dev);
    if (B->meta_dev) cudaFree(B->meta_dev);
    if (B->safety_d2_dev) cudaFree(B->safety_d2_dev);
    if (B->safety_lut_dev) cudaFree(B->safety_lut_dev);
    free(B->grid_host);
    free(B->meta_host);
    free(B);
}
extern "C" int mpp_map_batch_size(const mpp_map_batch *B) { return B ? B->n_maps : -1; }
extern "C" int mpp_map_batch_start(const mpp_map_batch *B, int k) { return (B && k >= 0 && k < B->n_maps) ? B->meta_host[k].start : -1; }
extern "C" int mpp_map_batch_target(const mpp_map_batch *B, int k) { return (B && k >= 0 && k < B->n_maps) ? B->meta_host[k].target : -1; }
extern "C" const uint32_t *mpp_map_batch_occ_bits(const mpp_map_batch *B, int *pitch_words) {
    if (!B) return nullptr;
    if (pitch_words) *pitch_words = B->pitch_words;
    return B->occ_dev;
}
extern "C" const uint8_t *mpp_map_batch_svalid(const mpp_map_batch *B) { return B ? B->svalid_dev : nullptr; }
extern "C" long long mpp_map_batch_obstacles(const mpp_map_batch *B) { return B ? B->n_obstacles : -1; }
