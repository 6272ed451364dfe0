// Standalone ICP ops (findNearest [ICP]:90-114, getTransform [ICP]:149-179) and the tuning switches of the
// batched kernel, which lives in b2s_icp_kernel.cuh (instantiated in b2s_icp_f32.cu / b2s_icp_f64.cu).
#include "b2s_icp_kernel.cuh"

namespace b2s {

// ICP.findNearest as a standalone op: src [n][2], tar [m][2] (point rows).  Targets are tiled
// through shared memory; each thread owns one source point.
constexpr int NN_TILE = 1024;

__global__ void __launch_bounds__(128)
nearest_kernel(const double *__restrict__ src_xy, int n, const double *__restrict__ tar_xy, int m,
               double *__restrict__ dist_out, int64_t *__restrict__ idx_out)
{
    __shared__ double2 tile[NN_TILE];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double sx = 0.0, sy = 0.0;
    if (i < n) {
        sx = src_xy[2 * i];
        sy = src_xy[2 * i + 1];
    }
    double best = INFINITY;
    long long arg = 0;
    for (int base = 0; base < m; base += NN_TILE) {
        const int cnt = min(NN_TILE, m - base);
        __syncthreads();
        for (int j = threadIdx.x; j < cnt; j += blockDim.x)
            tile[j] = make_double2(tar_xy[2 * (size_t)(base + j)], tar_xy[2 * (size_t)(base + j) + 1]);
        __syncthreads();
        for (int j = 0; j < cnt; ++j) {
            // the reference's own expression ([ICP]:102: np.linalg.norm of the difference), square root included:
            // sqrt merges neighbouring doubles, and the ties it creates go to the lower index
            const double d = ref_dist(sx - tile[j].x, sy - tile[j].y);
            if (d < best) {
                best = d;
                arg = base + j;
            }
        }
    }
    if (i < n) {
        dist_out[i] = (best == INFINITY) ? 0.0 : best;
        idx_out[i] = arg;
    }
}

// ICP.getTransform as a standalone op: one CTA, grid-stride over n row-matched points.
__global__ void __launch_bounds__(256)
rigid_fit_kernel(const double *__restrict__ src_xy, const double *__restrict__ tar_xy, int n,
                 double *__restrict__ T_out)
{
    __shared__ double scratch[4 * 32];
    double s4[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        s4[0] += src_xy[2 * i];
        s4[1] += src_xy[2 * i + 1];
        s4[2] += tar_xy[2 * i];
        s4[3] += tar_xy[2 * i + 1];
    }
    block_sum<4>(s4, scratch);
    const double inv = 1.0 / (double)n;
    const double cax = s4[0] * inv, cay = s4[1] * inv, cbx = s4[2] * inv, cby = s4[3] * inv;
    double w4[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double px = src_xy[2 * i] - cax, py = src_xy[2 * i + 1] - cay;
        const double qx = tar_xy[2 * i] - cbx, qy = tar_xy[2 * i + 1] - cby;
        w4[0] = fma(qx, px, w4[0]);
        w4[1] = fma(qx, py, w4[1]);
        w4[2] = fma(qy, px, w4[2]);
        w4[3] = fma(qy, py, w4[3]);
    }
    block_sum<4>(w4, scratch);
    if (threadIdx.x == 0) {
        double T[6];
        rotation_from_w(w4[0], w4[1], w4[2], w4[3], cax, cay, cbx, cby, T);
        T_out[0] = T[0]; T_out[1] = T[1]; T_out[2] = T[2];
        T_out[3] = T[3]; T_out[4] = T[4]; T_out[5] = T[5];
        T_out[6] = 0.0;  T_out[7] = 0.0;  T_out[8] = 1.0;
    }
}

int g_icp_src_per_thread = 0;  // 0: choose per problem size; 2..4 force (tuning hook)
int g_icp_layout = 2;          // point groups per warp: 2 balanced when that takes no extra group (default); 1 balanced; 0 strided (tuning hook)
int g_icp_prune = 4;           // exact search: 4 queued (default: both pruning tests, the surviving point x block pairs spread over the lanes);
                               // 2 collective, warp-level + per-lane pruning; 3 warp-level only; 1 per-lane only; 0 plain brute force
int g_icp_block = 0;           // targets per pruning block: 0 chooses per mode and scan size (8 up to 600 targets, 16 above); 8 / 16 / 32 force

// Points per thread: work is proportional to the register slots (threads x points per thread, idle ones included).
// Three is the measured optimum on B200 (360 and 1080 beams) and is taken unless it wastes more than 10 % over the
// leanest choice; then 4, then 2.
static int icp_points_per_thread(int n_src)
{
    if (g_icp_src_per_thread) return g_icp_src_per_thread;
    // a CTA must fit the register file: 65536 / 80 registers (R <= 3) is 819 threads, 65536 / 104 (R = 4) is 630
    // (the kernel's __maxnreg__); with a margin for the allocation granularity that is 768 / 576 threads, which is
    // what bounds the scan size to ICP_MAX_POINTS = 3 x 768 (the launch re-checks against the kernel's attributes)
    int slots[5] = {0, 0, 0, 0, 0}, least = 1 << 30;
    for (int c = 2; c <= 4; ++c) {
        int threads = ((((n_src + c - 1) / c) + 31) / 32) * 32;
        if (threads < 64) threads = 64;
        slots[c] = threads <= (c <= 3 ? 768 : 576) ? threads * c : (1 << 30);
        if (slots[c] < least) least = slots[c];
    }
    const int order[3] = {3, 4, 2};
    for (int k = 0; k < 3; ++k)
        if (slots[order[k]] < (1 << 30) && (long long)slots[order[k]] * 10 <= (long long)least * 11) return order[k];
    return 3;
}

int icp_dispatch(int n_src, int n_tar, int in_bytes, bool ranges, IcpInstance *out)
{
    B2S_REQUIRE(out, "b2s_icp_dispatch: null pointer");
    B2S_REQUIRE(n_src > 0 && n_tar > 0 && (in_bytes == 4 || in_bytes == 8) &&
                    (!ranges || (n_src == n_tar && in_bytes == 4)),
                ranges ? "b2s_icp_batch_ranges: bad sizes" : "b2s_icp_batch: bad sizes");
    B2S_REQUIRE(n_src <= ICP_MAX_POINTS, ranges ? "b2s_icp_batch_ranges: more than 2304 beams per scan is not supported"
                                                : "b2s_icp_batch: more than 2304 source points per scan is not supported");
    const int R = icp_points_per_thread(n_src);
    const int forced = (g_icp_block == 8 || g_icp_block == 16 || g_icp_block == 32) ? g_icp_block : 0;
    // queued search (icp_prune 4): block numbers travel in one byte, so at most QBLOCKS blocks, else the collective
    // search takes over; above QSUP_MIN blocks the warp test gets its second level (PRUNE 5)
    const int q8 = (n_tar + 7) / 8, q16 = (n_tar + 15) / 16;
    int P, B;
    if (ranges) {
        // the fused-ingestion form has the two default searches: queued, and the collective one of icp_prune 0..3
        const int blk = forced ? forced : (g_icp_prune == 4 || n_tar <= 600 ? 8 : 16);
        if (g_icp_prune == 4 && blk == 8 && q8 <= QBLOCKS) {
            P = q8 > QSUP_MIN ? 5 : 4;
            B = 8;
        } else if (g_icp_prune == 4 && q16 <= QBLOCKS) {
            P = q16 > QSUP_MIN ? 5 : 4;
            B = 16;
        } else {
            P = 2;
            B = blk;
        }
    } else {
        const int blk = forced ? forced
                               : (g_icp_prune == 4 ? 8 : g_icp_prune >= 2 ? (n_tar <= 600 ? 8 : 16) : (n_tar <= 600 ? 16 : 32));  // measured best per mode
        // the block bounds live in the staging area: [ceil(m/blk)] float4 must fit in 2*m*in_bytes
        const bool fits = (size_t)((n_tar + blk - 1) / blk) * 16 <= (size_t)2 * n_tar * in_bytes;
        if (!g_icp_prune || !fits) {
            P = 0;
            B = 16;
        } else if (g_icp_prune == 4 && blk == 8 && q8 <= QBLOCKS) {
            P = q8 > QSUP_MIN ? 5 : 4;
            B = 8;
        } else if (g_icp_prune == 4 && q16 <= QBLOCKS) {
            P = q16 > QSUP_MIN ? 5 : 4;
            B = 16;
        } else if (g_icp_prune >= 2) {  // 2 and 3, and 4 beyond the queue's block count
            P = g_icp_prune == 3 ? 3 : 2;
            B = blk;
        } else {
            P = 1;
            B = blk == 32 ? 32 : 16;
        }
    }
    int threads = ((((n_src + R - 1) / R) + 31) / 32) * 32;
    if (threads < 64) threads = 64;
    B2S_REQUIRE(threads <= 1024, ranges ? "b2s_icp_batch_ranges: too many beams per scan"
                                        : "b2s_icp_batch: too many source points per scan");
    const size_t smem = icp_smem_bytes(P, B, R, n_tar, (size_t)(ranges ? 1 : 2) * n_tar * in_bytes, threads);
    B2S_REQUIRE(smem <= 227 * 1024, ranges ? "b2s_icp_batch_ranges: too many beams for shared memory"
                                           : "b2s_icp_batch: n_tar too large for shared memory");
    *out = IcpInstance{R, P, B, threads, smem};
    return B2S_OK;
}

}  // namespace b2s

using namespace b2s;

extern "C" int b2s_nearest_f64(const double *src_xy, int n, const double *tar_xy, int m,
                               double *dist_out, int64_t *idx_out, void *stream)
{
    B2S_REQUIRE(n >= 0 && m >= 0, "b2s_nearest: negative size");
    if (n == 0) return B2S_OK;
    B2S_REQUIRE(src_xy && dist_out && idx_out && (tar_xy || m == 0), "b2s_nearest: null pointer");
    nearest_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(src_xy, n, tar_xy, m, dist_out, idx_out);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

extern "C" int b2s_icp_dispatch(int n_src, int n_tar, int in_bytes, int ranges, int *R, int *prune, int *nn_blk)
{
    B2S_REQUIRE(R && prune && nn_blk, "b2s_icp_dispatch: null pointer");
    IcpInstance ins;
    const int rc = icp_dispatch(n_src, n_tar, in_bytes, ranges != 0, &ins);
    if (rc != B2S_OK) return rc;
    *R = ins.R;
    *prune = ins.prune;
    *nn_blk = ins.nn_blk;
    return B2S_OK;
}

extern "C" int b2s_rigid_fit_f64(const double *src_xy, const double *tar_xy, int n, double *T_out,
                                 void *stream)
{
    B2S_REQUIRE(n > 0, "b2s_rigid_fit: need at least one point");
    B2S_REQUIRE(src_xy && tar_xy && T_out, "b2s_rigid_fit: null pointer");
    rigid_fit_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(src_xy, tar_xy, n, T_out);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}
