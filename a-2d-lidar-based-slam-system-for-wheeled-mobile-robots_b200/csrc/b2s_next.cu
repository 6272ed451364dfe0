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
//                 mean_error ([ICP]:75), ties to the lower index, composed with its candidate ([ICP]:185-190); for the
//                 coarse-to-fine form, the `keep` best coarse hypotheses per scan (radix select) and their rows.
//   track         hypotheses carried through consecutive scans: per stage the map observation's pose, the next
//                 prior moved by the odometry, the summed score; then the lowest finite joint score.
#include "b2s_common.cuh"

#include <math.h>

namespace b2s {

constexpr int CHAIN_THREADS = 1024;

// Exclusive prefix over a CTA of 1024 threads of one value per thread; returns this thread's offset, total in *total.
// scratch: 64 values of shared memory.  The offset is a sum of the values below this thread only: it is the inclusive
// value of the lane below, never inclusive minus own, so a NaN or inf of this thread cannot reach its own offset.
template <class V>
__device__ __forceinline__ V cta_exclusive_scan(V v, V *scratch, V *total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    V inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const V up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += up;
    }
    const V below = __shfl_up_sync(0xffffffffu, inc, 1);
    const V exc = lane ? below : V(0);
    if (lane == 31) scratch[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        V w = scratch[lane];  // CHAIN_THREADS / 32 == 32 warps
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const V up = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += up;
        }
        scratch[32 + lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const V before_warp = warp ? scratch[32 + warp - 1] : V(0);
    *total = scratch[63];
    __syncthreads();
    return before_warp + exc;
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
// KEPT: row j of scan k is candidate kept[k][j] (the survivors of relocalize_keep_kernel, ascending), so the lowest j
// among equal scores is also the lowest candidate; the candidate is reported and composed.
constexpr int SELECT_THREADS = 256;

__device__ __forceinline__ void select_better(double &bs, int &bh, double s, int h)
{
    if (h >= 0 && (bh < 0 || s < bs || (s == bs && h < bh))) {
        bs = s;
        bh = h;
    }
}

// [ICP]:185-190, the pose-chain step p (+) t of one transform t [9]: the relocalization's and the tracking's poses
__device__ __forceinline__ void pose_step(const double *p, const double *t, double *out)
{
    const double x = p[0], y = p[1], yaw = p[2];
    const double c = cos(yaw), s = sin(yaw);
    out[0] = x + c * t[2] - s * t[5];
    out[1] = y + s * t[2] + c * t[5];
    out[2] = yaw + atan2(t[3], t[0]);
}

template <bool KEPT>
__global__ void __launch_bounds__(SELECT_THREADS)
relocalize_select_kernel(const double *__restrict__ score, const double *__restrict__ T,
                         const double *__restrict__ cand, const int32_t *__restrict__ kept, int hyps,
                         int32_t *__restrict__ best_out, double *__restrict__ pose_out)
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
    const int bc = (KEPT && bh >= 0) ? kept[(size_t)k * hyps + bh] : bh;  // the winner's candidate
    best_out[k] = bc;
    double *pose = pose_out + 3 * (size_t)k;
    if (bh < 0) {
        pose[0] = pose[1] = pose[2] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    pose_step(cand + 3 * (size_t)bc, Tk + (size_t)bh * 9, pose);
}

// Pose tracking, the step after stage k's solves: thread h composes pose[h] = prior[h] (+) T[h], adds the stage's
// score to joint[h] (from 0.0 at stage 0, in ascending k) and keeps finite[h] only while the score, all nine entries
// of T and the pose stay finite; before the last stage it also writes the next prior, pose[h] (+) odo, into the pose
// rows the next stage's virtual scans read.  A track that went non-finite keeps running on whatever it holds.
constexpr int TRACK_THREADS = 256;

__global__ void __launch_bounds__(TRACK_THREADS)
track_step_kernel(const double *__restrict__ T, const double *__restrict__ score, const double *__restrict__ odo,
                  int hyps, int stage, const double *__restrict__ prior, double *__restrict__ pose,
                  double *__restrict__ next_prior, double *__restrict__ joint, int32_t *__restrict__ finite)
{
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= hyps) return;
    const double s = score[h];
    const double *t = T + (size_t)h * 9;
    bool fin = fabs(s) < INFINITY;  // false for NaN and +-inf
    for (int i = 0; i < 9; ++i) fin = fin && fabs(t[i]) < INFINITY;
    double q[3];
    pose_step(prior + 3 * (size_t)h, t, q);
    fin = fin && fabs(q[0]) < INFINITY && fabs(q[1]) < INFINITY && fabs(q[2]) < INFINITY;
    pose[3 * (size_t)h] = q[0];
    pose[3 * (size_t)h + 1] = q[1];
    pose[3 * (size_t)h + 2] = q[2];
    joint[h] = (stage == 0 ? 0.0 : joint[h]) + s;
    finite[h] = (stage == 0 || finite[h]) && fin;
    if (odo) pose_step(q, odo, next_prior + 3 * (size_t)h);
}

// Pose tracking, the selection: the smallest (joint, h) among the finite tracks, -1 when none is (one CTA).
constexpr int TRACK_SELECT_THREADS = 1024;

__global__ void __launch_bounds__(TRACK_SELECT_THREADS)
track_select_kernel(const double *__restrict__ joint, const int32_t *__restrict__ finite, int hyps,
                    int32_t *__restrict__ best_out)
{
    __shared__ double ws[TRACK_SELECT_THREADS / 32];
    __shared__ int wh[TRACK_SELECT_THREADS / 32];
    double bs = 0.0;
    int bh = -1;
    for (int h = threadIdx.x; h < hyps; h += blockDim.x)
        if (finite[h]) select_better(bs, bh, joint[h], h);
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
    *best_out = bh;
}

// Coarse-to-fine relocalization, the keep step: CTA k picks the `keep` best of scan k's `hyps` coarse hypotheses and
// writes their indices to kept[k][0..keep) in ascending order.  Each hypothesis gets a 64-bit key that orders like
// (finite score, with -0 == +0) and puts every non-finite hypothesis (score or any entry of T) above every finite one;
// the keep-th smallest key is found by a radix select of 8-bit digits (a 256-bin histogram in shared memory per
// digit, over the keys staged in `keys` [scans][hyps]), and the survivors are the keys below it plus, in ascending h,
// as many of the keys equal to it as are still missing.  That is the first `keep` of the strict order (key, h), the
// order of relocalize_select_kernel's finite rule followed by the non-finite hypotheses by h.
constexpr int KEEP_THREADS = 1024;  // cta_exclusive_scan's CTA

__device__ __forceinline__ unsigned long long keep_key(const double *__restrict__ s, const double *__restrict__ T, size_t h)
{
    bool finite = fabs(s[h]) < INFINITY;
    for (int i = 0; i < 9; ++i) finite = finite && fabs(T[h * 9 + i]) < INFINITY;
    if (!finite) return ~0ull;
    unsigned long long b = (unsigned long long)__double_as_longlong(s[h]);
    if (b == 0x8000000000000000ull) b = 0;  // -0.0 ties with +0.0
    return (b >> 63) ? ~b : b | 0x8000000000000000ull;  // negative: all bits flipped; positive: the sign bit set
}

__global__ void __launch_bounds__(KEEP_THREADS)
relocalize_keep_kernel(const double *__restrict__ score, const double *__restrict__ T, int hyps, int keep,
                       unsigned long long *__restrict__ keys, int32_t *__restrict__ kept)
{
    __shared__ unsigned int hist[256];
    __shared__ unsigned long long scratch[64];
    __shared__ unsigned int pick[2];  // the digit of this pass, the rank still wanted among keys with its prefix
    const int k = blockIdx.x, lane = threadIdx.x & 31;
    const size_t H = (size_t)hyps;
    const double *sk = score + (size_t)k * H, *Tk = T + (size_t)k * H * 9;
    unsigned long long *key = keys + (size_t)k * H;
    int32_t *out = kept + (size_t)k * keep;
    unsigned long long prefix = 0, mask = 0;
    unsigned int want = (unsigned int)keep;  // 1-based rank of the threshold among the keys that match prefix
    for (int shift = 56; shift >= 0; shift -= 8) {
        for (int i = threadIdx.x; i < 256; i += KEEP_THREADS) hist[i] = 0;
        __syncthreads();
        // warp-uniform trip count, so that every lane takes part in __match_any_sync
        for (size_t base = threadIdx.x - lane; base < H; base += KEEP_THREADS) {
            const size_t h = base + lane;
            unsigned long long v = 0;
            if (h < H) {
                if (shift == 56) key[h] = v = keep_key(sk, Tk, h);  // every later pass of this thread reads its own h
                else v = key[h];
            }
            const bool in = h < H && (v & mask) == prefix;
            const unsigned int d = in ? (unsigned int)(v >> shift) & 255u : 256u;
            const unsigned int peers = __match_any_sync(0xffffffffu, d);
            if (in && lane == __ffs(peers) - 1) atomicAdd(&hist[d], (unsigned int)__popc(peers));
        }
        __syncthreads();
        if (threadIdx.x < 32) {  // the digit whose bin holds rank `want`: lane l sums bins 8l .. 8l + 7
            unsigned int sum = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) sum += hist[8 * lane + i];
            unsigned int inc = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int up = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += up;
            }
            unsigned int before = inc - sum;
            if (before < want && want <= inc) {
                int d = 8 * lane;
                while (before + hist[d] < want) before += hist[d++];
                pick[0] = (unsigned int)d;
                pick[1] = want - before;
            }
        }
        __syncthreads();
        prefix |= (unsigned long long)pick[0] << shift;
        mask |= 255ull << shift;
        want = pick[1];
    }
    // prefix is the keep-th key: the keys below it survive, and the first `want` of the keys equal to it.  One
    // exclusive scan per tile of KEEP_THREADS hypotheses counts both (below: low word, equal: high word); a survivor's
    // slot is the number of survivors before it, below + min(equal, want).
    const unsigned int below_all = (unsigned int)keep - want;
    unsigned long long seen = 0;
    for (size_t base = 0; base < H; base += KEEP_THREADS) {
        const size_t h = base + threadIdx.x;
        const unsigned long long v = h < H ? key[h] : 0;
        const bool lt = h < H && v < prefix, eq = h < H && v == prefix;
        unsigned long long total;
        const unsigned long long before = seen + cta_exclusive_scan<unsigned long long>(
            (unsigned long long)lt | ((unsigned long long)eq << 32), scratch, &total);
        const unsigned int lt_before = (unsigned int)before, eq_before = (unsigned int)(before >> 32);
        if (lt || (eq && eq_before < want)) out[lt_before + min(eq_before, want)] = (int32_t)h;
        seen += total;
        if ((unsigned int)seen == below_all && (unsigned int)(seen >> 32) >= want) break;  // all survivors written
    }
}

// Rows of the refinement of a coarse-to-fine relocalization: pair p = k * keep + j gets the target row of candidate
// kept[p] (one of the `row`-double rows of `tar`, shared by every scan) and the source row of scan k.
__global__ void __launch_bounds__(256)
relocalize_gather_kernel(const double *__restrict__ tar, const double *__restrict__ src, const int32_t *__restrict__ kept,
                         size_t keep, size_t row, size_t pairs, double *__restrict__ tar_out, double *__restrict__ src_out)
{
    const size_t total = row * pairs;
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += (size_t)gridDim.x * blockDim.x) {
        const size_t p = j / row, i = j - p * row;
        tar_out[j] = tar[(size_t)kept[p] * row + i];
        src_out[j] = src[(p / keep) * row + i];
    }
}

int relocalize_gather(const double *tar, const double *src, const int32_t *kept, int scans, int keep, size_t row,
                      double *tar_out, double *src_out, cudaStream_t st)
{
    const size_t total = row * (size_t)scans * keep;
    if (total == 0) return B2S_OK;
    const size_t want = (total + 255) / 256, cap = (size_t)sm_count() * 16;
    relocalize_gather_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(tar, src, kept, (size_t)keep, row,
                                                                                  (size_t)scans * keep, tar_out, src_out);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
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
    relocalize_select_kernel<false><<<scans, SELECT_THREADS, 0, (cudaStream_t)stream>>>(score, T, candidates3, nullptr, hyps,
                                                                                        best_out, pose_out);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

extern "C" int b2s_relocalize_select_kept(const double *score, const double *T, const double *candidates3,
                                          const int32_t *kept, int scans, int keep, int32_t *best_out, double *pose_out,
                                          void *stream)
{
    B2S_REQUIRE(scans >= 0 && keep > 0, "b2s_relocalize_select_kept: bad sizes");
    if (scans == 0) return B2S_OK;
    B2S_REQUIRE(score && T && candidates3 && kept && best_out && pose_out, "b2s_relocalize_select_kept: null pointer");
    relocalize_select_kernel<true><<<scans, SELECT_THREADS, 0, (cudaStream_t)stream>>>(score, T, candidates3, kept, keep,
                                                                                       best_out, pose_out);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

extern "C" int b2s_relocalize_keep(const double *score, const double *T, int scans, int hyps, int keep, uint64_t *keys,
                                   int32_t *kept_out, void *stream)
{
    B2S_REQUIRE(scans >= 0 && hyps > 0 && keep > 0 && (long long)scans * hyps <= 0x7fffffffLL,
                "b2s_relocalize_keep: bad sizes");
    if (scans == 0) return B2S_OK;
    B2S_REQUIRE(score && T && keys && kept_out, "b2s_relocalize_keep: null pointer");
    relocalize_keep_kernel<<<scans, KEEP_THREADS, 0, (cudaStream_t)stream>>>(score, T, hyps, keep < hyps ? keep : hyps,
                                                                             (unsigned long long *)keys, kept_out);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

extern "C" int b2s_track_step(const double *T, const double *score, const double *odometry, int hyps, int stage,
                              const double *prior, double *pose, double *next_prior, double *joint, int32_t *finite,
                              void *stream)
{
    B2S_REQUIRE(hyps > 0 && stage >= 0, "b2s_track_step: bad sizes");
    B2S_REQUIRE(T && score && prior && pose && joint && finite, "b2s_track_step: null pointer");
    B2S_REQUIRE((odometry == nullptr) == (next_prior == nullptr), "b2s_track_step: odometry and next_prior go together");
    track_step_kernel<<<(unsigned)((hyps + TRACK_THREADS - 1) / TRACK_THREADS), TRACK_THREADS, 0, (cudaStream_t)stream>>>(
        T, score, odometry, hyps, stage, prior, pose, next_prior, joint, finite);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

extern "C" int b2s_track_select(const double *joint, const int32_t *finite, int hyps, int32_t *best_out, void *stream)
{
    B2S_REQUIRE(hyps > 0, "b2s_track_select: bad sizes");
    B2S_REQUIRE(joint && finite && best_out, "b2s_track_select: null pointer");
    track_select_kernel<<<1, TRACK_SELECT_THREADS, 0, (cudaStream_t)stream>>>(joint, finite, hyps, best_out);
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
