// Adjacent steps of the hot path (SURVEY.md section 8f): odometry pose chain, virtual scan.
//
//   pose chain    [ICP]:185-190 / W9 localization.py:79-83: x += cos(th) T02 - sin(th) T12, y += ..., th += atan2(T10, T00)
//                 over a stream of per-pair transforms -> a prefix sum of the yaw increments followed by a
//                 prefix sum of the rotated translations (one CTA, blocked scan).
//   virtual scan  W9 localization.py:128-150 (laserEstimation): min range per bearing bin over the static-map
//                 obstacle cells -> one thread per obstacle, atomicMin on the float64 bit pattern.  The batched form
//                 reduces each pose's bins in shared memory and can write them as the ICP's target cloud.
//   laserToNumpy  [ICP]:216-229 / [SLAM]:115-123 of float32 ranges into float64 points (the ICP's source cloud).
//   relocalize    the selection among map observations at many candidate poses: per scan the lowest finite
//                 mean_error ([ICP]:75), ties to the lower index, composed with its candidate ([ICP]:185-190).
#include "b2s_common.cuh"

#include <math.h>

namespace b2s {

constexpr int CHAIN_THREADS = 1024;

// Exclusive prefix over the CTA of one double per thread; returns this thread's offset, total in *total.
__device__ __forceinline__ double cta_exclusive_scan(double v, double *scratch, double *total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += up;
    }
    if (lane == 31) scratch[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        double w = scratch[lane];  // CHAIN_THREADS / 32 == 32 warps
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double up = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += up;
        }
        scratch[32 + lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const double before_warp = warp ? scratch[32 + warp - 1] : 0.0;
    *total = scratch[63];
    __syncthreads();
    return before_warp + inc - v;
}

__global__ void __launch_bounds__(CHAIN_THREADS)
pose_chain_kernel(const double *__restrict__ T, int pairs, double x0, double y0, double th0,
                  double *__restrict__ traj)
{
    __shared__ double scratch[64];
    const int tid = threadIdx.x;
    const int per = (pairs + CHAIN_THREADS - 1) / CHAIN_THREADS;
    const int lo = min(pairs, tid * per), hi = min(pairs, lo + per);
    // pass 1: yaw.  th_k = th0 + sum_{i<k} atan2(T10_i, T00_i)
    double part = 0.0;
    for (int k = lo; k < hi; ++k) part += atan2(T[9 * k + 3], T[9 * k + 0]);
    double total;
    double th = th0 + cta_exclusive_scan(part, scratch, &total);
    if (tid == 0) {
        traj[0] = x0;
        traj[1] = y0;
        traj[2] = th0;
    }
    // pass 2: position, each increment rotated by the yaw BEFORE the step ([ICP]:187-190)
    double px = 0.0, py = 0.0;
    double t2 = th;
    for (int k = lo; k < hi; ++k) {
        const double c = cos(t2), s = sin(t2);
        px += c * T[9 * k + 2] - s * T[9 * k + 5];
        py += s * T[9 * k + 2] + c * T[9 * k + 5];
        t2 += atan2(T[9 * k + 3], T[9 * k + 0]);
    }
    const double bx = x0 + cta_exclusive_scan(px, scratch, &total);
    const double by = y0 + cta_exclusive_scan(py, scratch, &total);
    double x = bx, y = by;
    for (int k = lo; k < hi; ++k) {
        const double c = cos(th), s = sin(th);
        x += c * T[9 * k + 2] - s * T[9 * k + 5];
        y += s * T[9 * k + 2] + c * T[9 * k + 5];
        th += atan2(T[9 * k + 3], T[9 * k + 0]);
        traj[3 * (k + 1)] = x;
        traj[3 * (k + 1) + 1] = y;
        traj[3 * (k + 1) + 2] = th;
    }
}

// One obstacle of laserEstimation (localization.py:137-146): its range and bearing bin seen from (x, y, yaw).  Both the
// single-pose and the batched kernel call this, so their bins cannot drift apart.  The _rn intrinsics keep the compiler
// from contracting the subtractions or the division with the last multiply of an inlined atan2 / hypot.  Returns false
// where int() would raise (NaN) or overflow, and for a NaN distance: such an obstacle never lowers a bin.
__device__ __forceinline__ bool vscan_bin(double ox, double oy, double x, double y, double yaw, double angle_min,
                                          double angle_increment, int beams, int &index, double &dist)
{
    dist = hypot(__dsub_rn(x, ox), __dsub_rn(y, oy));                                              // :138
    const double bin = __ddiv_rn(__dsub_rn(__dsub_rn(atan2(__dsub_rn(oy, y), __dsub_rn(ox, x)), angle_min), yaw),
                                 angle_increment);                                                 // :139
    if (!(fabs(bin) < 2.0e9) || !(dist == dist)) return false;
    index = (int)bin;   // truncation toward zero
    index %= beams;     // the two while loops, :141-144
    if (index < 0) index += beams;
    return true;
}

// distances are >= 0, so the IEEE bit patterns order like the values: the bins are min-reduced on the bits
__device__ __forceinline__ unsigned long long range_bits(double d) { return (unsigned long long)__double_as_longlong(d); }

// far_range into rows [scans][beams] of stride `stride` (the initial bins of the single-pose kernel and
// the merge target of the batched one)
__global__ void __launch_bounds__(256)
virtual_scan_fill_kernel(double *p, int scans, int beams, size_t stride, double far_range)
{
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= (size_t)scans * beams) return;
    const size_t k = j / beams;
    p[k * stride + (j - k * beams)] = far_range;
}

__global__ void __launch_bounds__(256)
virtual_scan_kernel(const double *__restrict__ obs_x, const double *__restrict__ obs_y, int count, double x,
                    double y, double yaw, double angle_min, double angle_increment, int beams,
                    double *__restrict__ ranges)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    int index;
    double dist;
    if (vscan_bin(obs_x[i], obs_y[i], x, y, yaw, angle_min, angle_increment, beams, index, dist))
        atomicMin(reinterpret_cast<unsigned long long *>(ranges) + index, range_bits(dist));
}

// Batched virtual scan: CTA (k, s) reduces obstacle slice s of pose k into bins in shared memory.  With one slice per
// pose (slices == 1) the CTA owns the pose and writes its ranges and target points itself.  Otherwise it merges only
// the bins it lowered below far_range into `merge` [scans][beams] (set to far_range beforehand) with a global
// atomicMin, and virtual_scan_points_kernel forms the points once every slice is done.  Rows of `merge` are
// merge_stride doubles apart: [scans][beams] ranges, or the x rows of the target [scans][2][beams].
constexpr int VSCAN_THREADS = 256;

__global__ void __launch_bounds__(VSCAN_THREADS)
virtual_scan_batch_kernel(const double *__restrict__ obs_x, const double *__restrict__ obs_y, int count, int per_slice,
                          const double *__restrict__ poses3, double angle_min, double angle_increment, int beams,
                          double far_range, const double2 *__restrict__ beam_cs, double *__restrict__ ranges,
                          double *__restrict__ tar_xy, double *__restrict__ merge, size_t merge_stride)
{
    extern __shared__ unsigned long long bins[];
    const int k = blockIdx.x;
    const double x = poses3[3 * k], y = poses3[3 * k + 1], yaw = poses3[3 * k + 2];
    const unsigned long long far = range_bits(far_range);
    for (int i = threadIdx.x; i < beams; i += VSCAN_THREADS) bins[i] = far;
    __syncthreads();
    const int c0 = blockIdx.y * per_slice, c1 = min(count, c0 + per_slice);
    for (int c = c0 + threadIdx.x; c < c1; c += VSCAN_THREADS) {
        int index;
        double dist;
        if (vscan_bin(obs_x[c], obs_y[c], x, y, yaw, angle_min, angle_increment, beams, index, dist))
            atomicMin(bins + index, range_bits(dist));
    }
    __syncthreads();
    if (merge) {
        unsigned long long *m = reinterpret_cast<unsigned long long *>(merge + (size_t)k * merge_stride);
        for (int i = threadIdx.x; i < beams; i += VSCAN_THREADS)
            if (bins[i] < far) atomicMin(m + i, bins[i]);
        return;
    }
    const size_t row = (size_t)k * beams;
    for (int i = threadIdx.x; i < beams; i += VSCAN_THREADS) {
        const double r = __longlong_as_double((long long)bins[i]);
        if (ranges) ranges[row + i] = r;
        if (tar_xy) {  // laserToNumpy: np.cos(a) * r, np.sin(a) * r -- one IEEE multiply each
            const double2 cs = beam_cs[i];
            tar_xy[2 * row + i] = __dmul_rn(cs.x, r);
            tar_xy[2 * row + beams + i] = __dmul_rn(cs.y, r);
        }
    }
}

// Points of the merged ranges (multi-slice path).  `ranges` may alias the x row of tar_xy: each thread reads its range
// before it writes the two coordinates.
__global__ void __launch_bounds__(256)
virtual_scan_points_kernel(const double *ranges, const double2 *__restrict__ beam_cs, int scans, int beams,
                           size_t range_stride, double *tar_xy)
{
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= (size_t)scans * beams) return;
    const size_t k = j / beams;
    const int i = (int)(j - k * beams);
    const double r = ranges[k * range_stride + i];
    const double2 cs = beam_cs[i];
    tar_xy[2 * k * beams + i] = __dmul_rn(cs.x, r);
    tar_xy[2 * k * beams + beams + i] = __dmul_rn(cs.y, r);
}

// laserToNumpy of raw float32 ranges into float64 points [scans][2][beams], with the arithmetic of the ICP kernel's
// RANGES form (b2s_icp_kernel.cuh, icp_batch_kernel's `point`): +inf -> clamp when clamp > 0, then one IEEE multiply.
__global__ void __launch_bounds__(256)
laser_points_kernel(const float *__restrict__ ranges, const double2 *__restrict__ beam_cs, double clamp, int scans,
                    int beams, double *__restrict__ xy)
{
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= (size_t)scans * beams) return;
    const size_t k = j / beams;
    const int i = (int)(j - k * beams);
    double r = (double)ranges[j];
    if (clamp > 0.0 && r == INFINITY) r = clamp;  // [SLAM]:119 (only +inf compares equal)
    const double2 cs = beam_cs[i];
    xy[2 * k * beams + i] = __dmul_rn(cs.x, r);
    xy[2 * k * beams + beams + i] = __dmul_rn(cs.y, r);
}

// `copies` consecutive copies of one row of `row` doubles: the source cloud of a scan for every hypothesis of a
// relocalization (the ICP kernel reads pair p's source at p * row).
__global__ void __launch_bounds__(256)
replicate_row_kernel(const double *__restrict__ src, size_t row, size_t copies, double *__restrict__ dst)
{
    const size_t total = row * copies;
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += (size_t)gridDim.x * blockDim.x)
        dst[j] = src[j % row];
}

// Relocalization selection: CTA k reduces the scores of scan k's hypotheses to the smallest (score, h) among those
// whose score and transform are finite, then composes the winner's pose.  (score, h) with the lower h winning equal
// scores is a strict total order in which every h occurs once, so the minimum is one element whatever the order of
// the comparisons: the result does not depend on the CTA's thread count or on how the reduction is cut.
constexpr int SELECT_THREADS = 256;

__device__ __forceinline__ void select_better(double &bs, int &bh, double s, int h)
{
    if (h >= 0 && (bh < 0 || s < bs || (s == bs && h < bh))) {
        bs = s;
        bh = h;
    }
}

__global__ void __launch_bounds__(SELECT_THREADS)
relocalize_select_kernel(const double *__restrict__ score, const double *__restrict__ T,
                         const double *__restrict__ cand, int hyps, int32_t *__restrict__ best_out,
                         double *__restrict__ pose_out)
{
    __shared__ double ws[SELECT_THREADS / 32];
    __shared__ int wh[SELECT_THREADS / 32];
    const int k = blockIdx.x;
    const double *sk = score + (size_t)k * hyps;
    const double *Tk = T + (size_t)k * hyps * 9;
    double bs = 0.0;
    int bh = -1;  // -1: nothing finite yet
    for (int h = threadIdx.x; h < hyps; h += blockDim.x) {
        const double s = sk[h];
        bool finite = fabs(s) < INFINITY;  // false for NaN and +-inf
        for (int i = 0; i < 9; ++i) finite = finite && fabs(Tk[(size_t)h * 9 + i]) < INFINITY;
        if (finite) select_better(bs, bh, s, h);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double os = __shfl_xor_sync(0xffffffffu, bs, o);
        const int oh = __shfl_xor_sync(0xffffffffu, bh, o);
        select_better(bs, bh, os, oh);
    }
    if (lane == 0) {
        ws[warp] = bs;
        wh[warp] = bh;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) select_better(bs, bh, ws[w], wh[w]);
    best_out[k] = bh;
    double *pose = pose_out + 3 * (size_t)k;
    if (bh < 0) {
        pose[0] = pose[1] = pose[2] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    // [ICP]:185-190, the pose-chain step of one transform
    const double *t = Tk + (size_t)bh * 9;
    const double x = cand[3 * (size_t)bh], y = cand[3 * (size_t)bh + 1], yaw = cand[3 * (size_t)bh + 2];
    const double c = cos(yaw), s = sin(yaw);
    pose[0] = x + c * t[2] - s * t[5];
    pose[1] = y + s * t[2] + c * t[5];
    pose[2] = yaw + atan2(t[3], t[0]);
}

int replicate_row(const double *src, size_t row, size_t copies, double *dst, cudaStream_t st)
{
    const size_t total = row * copies;
    if (total == 0) return B2S_OK;
    const size_t want = (total + 255) / 256, cap = (size_t)sm_count() * 16;
    replicate_row_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(src, row, copies, dst);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

// Slices per pose: one CTA per pose when the poses alone fill the device a few times over; otherwise the obstacles are
// cut into slices of at least VSCAN_MIN_SLICE cells so that a small batch over a large map still spreads over every SM.
constexpr int VSCAN_MIN_SLICE = 1024;

static int vscan_slices(int count, int scans)
{
    const long long want_ctas = (long long)sm_count() * 8;
    if (count <= VSCAN_MIN_SLICE || scans >= want_ctas) return 1;
    const long long by_size = (count + VSCAN_MIN_SLICE - 1) / VSCAN_MIN_SLICE;
    const long long by_fill = (want_ctas + scans - 1) / scans;
    return (int)(by_size < by_fill ? by_size : by_fill);
}

int laser_points(const float *ranges, const double *beam_cs, double clamp, int scans, int beams, double *xy,
                 cudaStream_t st)
{
    const size_t total = (size_t)scans * beams;
    if (total == 0) return B2S_OK;
    laser_points_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(ranges, reinterpret_cast<const double2 *>(beam_cs),
                                                                        clamp, scans, beams, xy);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

}  // namespace b2s

using namespace b2s;

extern "C" int b2s_pose_chain(const double *T, int pairs, double x0, double y0, double th0, double *traj,
                              void *stream)
{
    B2S_REQUIRE(pairs >= 0 && traj && (T || pairs == 0), "b2s_pose_chain: bad arguments");
    pose_chain_kernel<<<1, CHAIN_THREADS, 0, (cudaStream_t)stream>>>(T, pairs, x0, y0, th0, traj);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

extern "C" int b2s_virtual_scan(const double *obs_x, const double *obs_y, int count, double x, double y,
                                double yaw, double angle_min, double angle_increment, int beams,
                                double far_range, double *ranges, void *stream)
{
    B2S_REQUIRE(count >= 0 && beams > 0 && ranges && (count == 0 || (obs_x && obs_y)), "b2s_virtual_scan: bad arguments");
    B2S_REQUIRE(angle_increment != 0.0 && angle_increment == angle_increment, "b2s_virtual_scan: angle_increment");
    cudaStream_t st = (cudaStream_t)stream;
    virtual_scan_fill_kernel<<<(beams + 255) / 256, 256, 0, st>>>(ranges, 1, beams, beams, far_range);
    B2S_CUDA(cudaGetLastError());
    if (count > 0) {
        virtual_scan_kernel<<<(count + 255) / 256, 256, 0, st>>>(obs_x, obs_y, count, x, y, yaw, angle_min,
                                                                 angle_increment, beams, ranges);
        B2S_CUDA(cudaGetLastError());
    }
    return B2S_OK;
}

extern "C" int b2s_virtual_scan_batch(const double *obs_x, const double *obs_y, int count, const double *poses3, int scans,
                                      double angle_min, double angle_increment, int beams, double far_range,
                                      const double *beam_cs, double *ranges, double *tar_xy, void *stream)
{
    B2S_REQUIRE(count >= 0 && scans >= 0 && beams > 0, "b2s_virtual_scan_batch: bad sizes");
    B2S_REQUIRE(beams <= B2S_VSCAN_MAX_BEAMS, "b2s_virtual_scan_batch: more than 6144 beams per scan is not supported");
    B2S_REQUIRE((count == 0 || (obs_x && obs_y)) && (scans == 0 || poses3) && (ranges || tar_xy),
                "b2s_virtual_scan_batch: null pointer");
    B2S_REQUIRE(!tar_xy || (beam_cs && (uintptr_t)beam_cs % 16 == 0),
                "b2s_virtual_scan_batch: tar_xy needs a 16-byte aligned beam table");
    B2S_REQUIRE(angle_increment != 0.0 && angle_increment == angle_increment, "b2s_virtual_scan_batch: angle_increment");
    if (scans == 0) return B2S_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int slices = vscan_slices(count, scans);
    const int per_slice = count > 0 ? (count + slices - 1) / slices : 0;
    const size_t smem = (size_t)beams * sizeof(unsigned long long);
    const double2 *cs = reinterpret_cast<const double2 *>(beam_cs);
    if (slices == 1) {
        virtual_scan_batch_kernel<<<dim3(scans, 1), VSCAN_THREADS, smem, st>>>(obs_x, obs_y, count, per_slice, poses3, angle_min,
                                                                               angle_increment, beams, far_range, cs, ranges,
                                                                               tar_xy, nullptr, 0);
        B2S_CUDA(cudaGetLastError());
        return B2S_OK;
    }
    // merged ranges go to `ranges`, or without it to the x rows of tar_xy, which the points kernel then overwrites
    double *merge = ranges ? ranges : tar_xy;
    const size_t stride = ranges ? (size_t)beams : (size_t)2 * beams;
    const size_t total = (size_t)scans * beams;
    const unsigned blocks = (unsigned)((total + 255) / 256);
    virtual_scan_fill_kernel<<<blocks, 256, 0, st>>>(merge, scans, beams, stride, far_range);
    B2S_CUDA(cudaGetLastError());
    virtual_scan_batch_kernel<<<dim3(scans, slices), VSCAN_THREADS, smem, st>>>(obs_x, obs_y, count, per_slice, poses3, angle_min,
                                                                                angle_increment, beams, far_range, cs, nullptr,
                                                                                nullptr, merge, stride);
    B2S_CUDA(cudaGetLastError());
    if (tar_xy) {
        virtual_scan_points_kernel<<<blocks, 256, 0, st>>>(merge, cs, scans, beams, stride, tar_xy);
        B2S_CUDA(cudaGetLastError());
    }
    return B2S_OK;
}

extern "C" int b2s_relocalize_select(const double *score, const double *T, const double *candidates3, int scans, int hyps,
                                     int32_t *best_out, double *pose_out, void *stream)
{
    B2S_REQUIRE(scans >= 0 && hyps > 0, "b2s_relocalize_select: bad sizes");
    if (scans == 0) return B2S_OK;
    B2S_REQUIRE(score && T && candidates3 && best_out && pose_out, "b2s_relocalize_select: null pointer");
    relocalize_select_kernel<<<scans, SELECT_THREADS, 0, (cudaStream_t)stream>>>(score, T, candidates3, hyps, best_out,
                                                                                 pose_out);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

// Host-buffer forms (the calls scan.py makes).
extern "C" int b2s_pose_chain_host(const double *T, int pairs, double x0, double y0, double th0, double *traj)
{
    B2S_REQUIRE(pairs >= 0 && traj && (T || pairs == 0), "b2s_pose_chain_host: bad arguments");
    ScratchPool *sp = scratch_pool();
    if (!sp) return cuda_fail(cudaErrorUnknown, "b2s_pose_chain_host: no device");
    int rc;
    if ((rc = sp->a.reserve((size_t)(pairs > 0 ? pairs : 1) * 72))) return rc;
    if ((rc = sp->b.reserve((size_t)(pairs + 1) * 24))) return rc;
    if (pairs > 0) B2S_CUDA(cudaMemcpyAsync(sp->a.p, T, (size_t)pairs * 72, cudaMemcpyHostToDevice, cudaStreamPerThread));
    if ((rc = b2s_pose_chain((const double *)sp->a.p, pairs, x0, y0, th0, (double *)sp->b.p, cudaStreamPerThread))) return rc;
    B2S_CUDA(cudaMemcpyAsync(traj, sp->b.p, (size_t)(pairs + 1) * 24, cudaMemcpyDeviceToHost, cudaStreamPerThread));
    B2S_CUDA(cudaStreamSynchronize(cudaStreamPerThread));
    return B2S_OK;
}

extern "C" int b2s_virtual_scan_host(const double *obs_x, const double *obs_y, int count, double x, double y,
                                     double yaw, double angle_min, double angle_increment, int beams,
                                     double far_range, double *ranges)
{
    B2S_REQUIRE(count >= 0 && beams > 0 && ranges && (count == 0 || (obs_x && obs_y)), "b2s_virtual_scan_host: bad arguments");
    ScratchPool *sp = scratch_pool();
    if (!sp) return cuda_fail(cudaErrorUnknown, "b2s_virtual_scan_host: no device");
    const size_t ob = (size_t)(count > 0 ? count : 1) * 8;
    int rc;
    if ((rc = sp->a.reserve(ob))) return rc;
    if ((rc = sp->b.reserve(ob))) return rc;
    if ((rc = sp->c.reserve((size_t)beams * 8))) return rc;
    if (count > 0) {
        B2S_CUDA(cudaMemcpyAsync(sp->a.p, obs_x, (size_t)count * 8, cudaMemcpyHostToDevice, cudaStreamPerThread));
        B2S_CUDA(cudaMemcpyAsync(sp->b.p, obs_y, (size_t)count * 8, cudaMemcpyHostToDevice, cudaStreamPerThread));
    }
    if ((rc = b2s_virtual_scan((const double *)sp->a.p, (const double *)sp->b.p, count, x, y, yaw, angle_min, angle_increment,
                               beams, far_range, (double *)sp->c.p, cudaStreamPerThread)))
        return rc;
    B2S_CUDA(cudaMemcpyAsync(ranges, sp->c.p, (size_t)beams * 8, cudaMemcpyDeviceToHost, cudaStreamPerThread));
    B2S_CUDA(cudaStreamSynchronize(cudaStreamPerThread));
    return B2S_OK;
}

// ---------------------------------------------------------------------------------------------
// Same-run FP64 issue peak (bench.py quotes the ICP kernel against it): 8 independent DFMA chains per thread.
namespace b2s {
__global__ void __launch_bounds__(256)
fp64_peak_kernel(double *out, int iters, double a, double b)
{
    double v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = (double)(threadIdx.x + k);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = fma(v[k], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += v[k];
    if (s == 123.456) out[0] = s;  // never true; keeps the chains alive
}
}  // namespace b2s

extern "C" int b2s_measure_fp64_peak(double *tflops_out)
{
    B2S_REQUIRE(tflops_out, "b2s_measure_fp64_peak: null pointer");
    double *d = nullptr;
    B2S_CUDA(cudaMalloc((void **)&d, 8));
    cudaEvent_t e0, e1;
    B2S_CUDA(cudaEventCreate(&e0));
    B2S_CUDA(cudaEventCreate(&e1));
    const int blocks = sm_count() * 8, iters = 4096;
    fp64_peak_kernel<<<blocks, 256>>>(d, iters, 0.999999, 1e-9);  // warm-up
    B2S_CUDA(cudaEventRecord(e0));
    fp64_peak_kernel<<<blocks, 256>>>(d, iters, 0.999999, 1e-9);
    B2S_CUDA(cudaEventRecord(e1));
    B2S_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    B2S_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    *tflops_out = 2.0 * 8.0 * iters * 256.0 * blocks / (ms * 1e-3) / 1e12;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    return B2S_OK;
}
