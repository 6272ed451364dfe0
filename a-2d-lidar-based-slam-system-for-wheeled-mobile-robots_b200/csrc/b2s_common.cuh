// Shared device/host helpers for the b2slam kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "b2slam.h"

namespace b2s {

void set_error(const char *fmt, ...);

inline int cuda_fail(cudaError_t e, const char *what)
{
    set_error("%s: %s", what, cudaGetErrorString(e));
    return B2S_ERR_CUDA;
}

#define B2S_CUDA(call)                                      \
    do {                                                    \
        cudaError_t e__ = (call);                           \
        if (e__ != cudaSuccess) return ::b2s::cuda_fail(e__, #call); \
    } while (0)

#define B2S_REQUIRE(cond, msg)                  \
    do {                                        \
        if (!(cond)) {                          \
            ::b2s::set_error("%s", msg);        \
            return B2S_ERR_INVALID_ARG;         \
        }                                       \
    } while (0)

int sm_count();

constexpr int ICP_MAX_POINTS = 2304;  // source points per scan of the ICP kernel; see icp_points_per_thread

// laserToNumpy of raw ranges [scans][beams] into float64 points [scans][2][beams] (b2s_next.cu); beam_cs [beams][2]
// 16-byte aligned, clamp > 0 replaces +inf.  The points are those the ICP kernel's fused form makes from the ranges.
int laser_points(const float *ranges, const double *beam_cs, double clamp, int scans, int beams, double *xy,
                 cudaStream_t stream);
// `copies` consecutive copies of the `row` doubles at src into dst (b2s_next.cu).
int replicate_row(const double *src, size_t row, size_t copies, double *dst, cudaStream_t stream);

// Growable device / pinned-host staging buffer.
struct Buf {
    void *p = nullptr;
    size_t cap = 0;
    bool pinned = false;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return B2S_OK;
        release();
        size_t want = bytes + bytes / 4;
        cudaError_t e = pinned ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            p = nullptr;
            cap = 0;
            set_error("allocation of %zu bytes failed: %s", want, cudaGetErrorString(e));
            return e == cudaErrorMemoryAllocation ? B2S_ERR_NOMEM : B2S_ERR_CUDA;
        }
        cap = want;
        return B2S_OK;
    }
    void release()
    {
        if (p) {
            if (pinned) cudaFreeHost(p); else cudaFree(p);
        }
        p = nullptr;
        cap = 0;
    }
};

// Per-thread, per-device scratch for the small host-buffer calls (pose chain, virtual scan, Bresenham paths): they are
// made once per scan by a node, so their device buffers are kept and grown instead of cudaMalloc'ed per call.
// Never freed (the CUDA context may be gone by the time thread-local destructors run).
struct ScratchPool {
    int device = -1;
    Buf a, b, c;
};
ScratchPool *scratch_pool();  // bound to the calling thread's current device; nullptr on a CUDA error


// Dirty-tile bookkeeping of the ray-cast workspace: one byte per 64 x 64-cell tile of the grid.
constexpr int GRID_TILE = 64;
constexpr int GRID_WS_HEADER = 64;
inline __host__ __device__ int grid_tiles(int w) { return (w + GRID_TILE - 1) / GRID_TILE; }
inline size_t grid_dirty_bytes(int xw, int yw)
{
    return (((size_t)grid_tiles(xw) * grid_tiles(yw)) + 255) & ~(size_t)255;
}

int grid_raycast_signed(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m, double off_x,
                        double off_y, const void *ox, const void *oy, const void *cx, const void *cy, bool is_f64,
                        int scans, int beams, int32_t *counters, void *workspace, int sign, void *stream,
                        bool fold = true);
int grid_finalize_dirty(const int32_t *hit, const int32_t *miss, int xw, int yw, double w_hit, double w_miss,
                        double thresh, void *workspace, int8_t *pmap, int8_t *packed, int32_t *tile_ids,
                        int32_t *counter, int cap, void *stream);
int grid_raycast_ranges_signed(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m, double off_x,
                               double off_y, const float *ranges, const double *pose4, const double *beam_cs,
                               double clamp, int scans, int beams, int32_t *counters, void *workspace, int sign,
                               void *stream, bool fold = true);
// fold = false leaves the y-major visits of this launch in the transposed scratch plane (and its bounding box in
// the workspace header): a caller that ray-casts a batch as several launches folds once, with the last of them.

// ---------------------------------------------------------------- warp / block reductions

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum K doubles over the whole CTA; every thread returns the same totals, accumulated in a
// fixed order (warp butterfly, then warps in index order) so results are run-to-run identical.
// scratch: K * 32 doubles of shared memory.  Contains two __syncthreads().
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double *scratch)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const double w = warp_sum(v[k]);
        if (lane == 0) scratch[k * 32 + warp] = w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double t = 0.0;
        for (int w = 0; w < nwarps; ++w) t += scratch[k * 32 + w];
        v[k] = t;
    }
    __syncthreads();
}

// ---------------------------------------------------------------- 1-D bulk async copy (TMA)

__device__ __forceinline__ uint32_t smem_addr(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
}

__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)),
                 "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_addr(bar)),
        "r"(parity)
        : "memory");
}

// global -> shared bulk copy; dst, src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_addr(dst)),
        "l"(src), "r"(bytes), "r"(smem_addr(bar))
        : "memory");
}

}  // namespace b2s
