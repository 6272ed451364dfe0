// Batched 2-D point-to-point ICP: one CTA per scan pair, whole iteration loop on chip.
//
// Replaces ICP.process ([ICP]:38-88), findNearest ([ICP]:90-114), getTransform ([ICP]:149-179).
//
// Per pair the kernel reads 2*(N+M) coordinates once (target rows staged into shared memory
// with a 1-D bulk async copy + mbarrier), then runs up to max_iter iterations of
//   nearest neighbour               (exact: the index of the N*M brute force with strict '<' in ascending j, i.e.
//                                    the lowest index wins ties like the reference loop, found with a warp-level
//                                    and a per-lane block-pruning test in front.  PRUNE = 4 / 5, the default, queues
//                                    the (point, block) pairs that survive both tests and spreads them over the lanes;
//                                    PRUNE = 1..3 evaluate a surviving block with the whole warp; 0 is the brute force)
//   centroid + 2x2 cross-covariance (ONE reduction about fixed shifts; the reference centres, then multiplies)
//   closed-form proper rotation     ((c, s) = (W00+W11, W10-W01) / norm == U.Vt with the W9 reflection fix)
//   src <- T.src, mean-error stop rule
// and the final re-fit of the original source onto the moved source ([ICP]:81).
//
// Numerics: everything is float64, like the reference.  B200 (sm_100a) issues FP64 at half the
// FP32 rate, and an FP32 search would need a second-best tracker plus a float64 re-check of
// near ties to keep correspondences identical, which costs about the same issue slots; see
// DESIGN.md "ICP numerics".  Source points live in registers (R per thread) for the whole solve (the queued search
// keeps a copy of the moved points in shared memory); targets live in shared memory as double2.
//
// This header holds the kernel and its launch logic; b2s_icp_f32.cu / b2s_icp_f64.cu instantiate it per input
// type (two translation units so the instances compile in parallel).
#pragma once
#include "b2s_common.cuh"

#include <math.h>

namespace b2s {

#ifndef B2S_ICP_REGS_BLK8
#define B2S_ICP_REGS_BLK8 72
#endif
#ifndef B2S_ICP_REGS_BLK16
#define B2S_ICP_REGS_BLK16 80
#endif

constexpr int FIT_SUMS = 9;
constexpr int NN_CHAINS = 4;
constexpr int SUM_PAD = 10;                          // doubles per warp slot (9 sums, padded for 16-byte loads)
// Bytes of the staging area: the input rows as they come (`in_bytes`), later reused for the block bounds (a float4
// per block); rounded to 16.
__host__ __device__ inline size_t icp_stage_bytes(size_t in_bytes, int nblk)
{
    const size_t b = ((size_t)nblk + (nblk + 31) / 32) * 16;  // + one bound per 32 blocks (queued search)
    return ((in_bytes > b ? in_bytes : b) + 15) & ~(size_t)15;
}

// Reduction scratch of a CTA of `nwarps` warps, in doubles: two buffers (alternating calls) of nwarps x SUM_PAD for
// cta_sum9, and 4 x 32 for the block_sum<4> of the set-up.
__host__ __device__ inline int icp_scratch_doubles(int nwarps)
{
    const int a = 2 * nwarps * SUM_PAD;
    return a > 128 ? a : 128;
}

// Sum of 8 values over the warp with 9 shuffles instead of 40: at offsets 16, 8, 4 every lane hands the half of
// its values it is not responsible for to its partner and keeps the other half, so the value count halves while
// the lane count doubles; two plain butterfly steps finish.  Afterwards lane l holds the warp total of value
// (l >> 2) & 7.  Fixed order, hence run-to-run identical.
__device__ __forceinline__ double warp_sum8_transposed(const double (&v)[8], int lane)
{
    const bool up16 = lane & 16, up8 = lane & 8, up4 = lane & 4;
    double a[4], b[2];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const double send = up16 ? v[i] : v[i + 4], keep = up16 ? v[i + 4] : v[i];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const double send = up8 ? a[i] : a[i + 2], keep = up8 ? a[i + 2] : a[i];
        b[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    const double send = up4 ? b[0] : b[1], keep = up4 ? b[1] : b[0];
    double c = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    c += __shfl_xor_sync(0xffffffffu, c, 2);
    c += __shfl_xor_sync(0xffffffffu, c, 1);
    return c;
}

// Sum FIT_SUMS doubles over the CTA; every thread returns the same totals (warps added in index order).
// ONE barrier per call: consecutive calls alternate between two scratch buffers (`phase`), so the next call's
// writes cannot overtake this call's reads.
__device__ __forceinline__ void cta_sum9(double (&v)[FIT_SUMS], double *scratch, int &phase)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps = (blockDim.x + 31) >> 5;
    double *buf = scratch + phase * (nwarps * SUM_PAD);
    phase ^= 1;
    const double v8[8] = {v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]};
    const double t = warp_sum8_transposed(v8, lane);
    const double last = warp_sum(v[8]);
    if ((lane & 3) == 0) buf[warp * SUM_PAD + ((lane >> 2) & 7)] = t;
    if (lane == 1) buf[warp * SUM_PAD + 8] = last;
    __syncthreads();
    if (nwarps <= 4) {
        // few warps: every thread adds the columns itself (nine independent chains, shortest latency; this sits
        // on the critical path right after the barrier)
#pragma unroll
        for (int k = 0; k < FIT_SUMS; ++k) v[k] = 0.0;
        for (int w = 0; w < nwarps; ++w) {
            const double2 *row = reinterpret_cast<const double2 *>(buf + w * SUM_PAD);
            const double2 p0 = row[0], p1 = row[1], p2 = row[2], p3 = row[3], p4 = row[4];
            v[0] += p0.x; v[1] += p0.y; v[2] += p1.x; v[3] += p1.y; v[4] += p2.x;
            v[5] += p2.y; v[6] += p3.x; v[7] += p3.y; v[8] += p4.x;
        }
    } else {
        // many warps: lane k adds up column k (1 load + 1 add per warp instead of 5 + 9), then the nine totals
        // are broadcast.  Both forms add the warps in index order.
        double acc = 0.0;
        if (lane < FIT_SUMS) {
#pragma unroll 4
            for (int w = 0; w < nwarps; ++w) acc += buf[w * SUM_PAD + lane];
        }
#pragma unroll
        for (int k = 0; k < FIT_SUMS; ++k) v[k] = __shfl_sync(0xffffffffu, acc, k);
    }
}

// Closed-form Kabsch for row-matched sets given centred sums; returns T (row-major 2x3 part).
__device__ __forceinline__ void rotation_from_w(double w00, double w01, double w10, double w11,
                                                double cax, double cay, double cbx, double cby,
                                                double (&T)[6])
{
    const double cc = w00 + w11, ss = w10 - w01;
    // (c, s) = (cc, ss) / |(cc, ss)|.  Every thread of the CTA evaluates this after each reduction, so the common
    // case takes one reciprocal square root (<= 2 ulp on c and s, far inside the 1e-9 the tests hold) instead of
    // hypot + two divisions; sums outside the safely squarable range take the careful path.
    const double h2 = fma(cc, cc, ss * ss);
    double c = 1.0, s = 0.0;
    if (h2 > 1e-280 && h2 < 1e280) {
        const double inv = rsqrt(h2);
        c = cc * inv;
        s = ss * inv;
    } else {
        const double h = hypot(cc, ss);
        if (h > 0.0) {
            c = cc / h;
            s = ss / h;
        }
    }
    T[0] = c;
    T[1] = -s;
    T[2] = cbx - (c * cax - s * cay);
    T[3] = s;
    T[4] = c;
    T[5] = cby - (s * cax + c * cay);
}

// getTransform ([ICP]:149-179) over the CTA for points held in registers: a[r] -> b[r].
//
// The reference centres both sets on their means and then forms W = BB^T.AA, which needs two
// reductions.  Here every coordinate is taken relative to a FIXED per-pair shift close to the
// centroids (sa, sb: the centroids of the original source / of the target scan), the first and
// second moments are reduced together in ONE block reduction, and the exact identity
//     sum (b-cb)(a-ca)^T = sum (b-sb)(a-sa)^T - n (cb-sb)(ca-sa)^T
// removes the offset.  Because |c - s| is of the order of the scan-to-scan motion while the spread
// of a scan is metres, the subtracted term is ~1e-3 of W and costs no accuracy (the parity tests hold
// the result to 1e-9 of the reference).  `extra` rides along in the same reduction (the distance sum).
template <int R>
__device__ __forceinline__ void cta_rigid_fit(const double (&ax)[R], const double (&ay)[R],
                                              const double (&bx)[R], const double (&by)[R], int count,
                                              int n, double sax, double say, double sbx, double sby,
                                              double &extra, double *scratch, int &phase, double (&T)[6])
{
    double v[FIT_SUMS];
#pragma unroll
    for (int k = 0; k < FIT_SUMS; ++k) v[k] = 0.0;
#pragma unroll
    for (int r = 0; r < R; ++r)
        if (r < count) {
            const double px = ax[r] - sax, py = ay[r] - say;
            const double qx = bx[r] - sbx, qy = by[r] - sby;
            v[0] += px;
            v[1] += py;
            v[2] += qx;
            v[3] += qy;
            v[4] = fma(qx, px, v[4]);  // W = BB^T . AA  ([ICP]:160)
            v[5] = fma(qx, py, v[5]);
            v[6] = fma(qy, px, v[6]);
            v[7] = fma(qy, py, v[7]);
        }
    v[8] = extra;
    cta_sum9(v, scratch, phase);
    const double inv = 1.0 / (double)n;
    const double mpx = v[0] * inv, mpy = v[1] * inv, mqx = v[2] * inv, mqy = v[3] * inv;
    const double w00 = v[4] - v[2] * mpx, w01 = v[5] - v[2] * mpy;
    const double w10 = v[6] - v[3] * mpx, w11 = v[7] - v[3] * mpy;
    (void)mqx;
    (void)mqy;
    rotation_from_w(w00, w01, w10, w11, sax + mpx, say + mpy, sbx + mqx, sby + mqy, T);
    extra = v[8];
}

// An upper bound of sqrt(x) for the pruning radii, x >= 0 in float32: the approximate square root (one MUFU, relative
// error <= 2^-22 by the PTX ISA, subnormal inputs flushed to zero) times 1 + 2^-20, plus more than the root of the
// largest flushed input.  Like the rounded-up exact root it replaces (a range check, a branch and six instructions),
// this only widens what the search looks at; inf stays inf and NaN stays NaN, which make every skip test false.
// x << s with PTX semantics: shift counts above 31 give 0 (the C++ operator leaves them undefined).
__device__ __forceinline__ unsigned shl_sat(unsigned x, unsigned s)
{
    unsigned r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(s));
    return r;
}

__device__ __forceinline__ float sqrt_up(float x)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return fmaf(r, 1.000001f, 2e-19f);
}

// ---------------------------------------------------------------- the reference's distance and its ties
//
// findNearest orders candidates by np.linalg.norm(src[i] - tar[j]) with a strict '<' in ascending j ([ICP]:99-106).
// NumPy evaluates that norm as sqrt(x.dot(x)), the dot product through the BLAS ddot whose scalar tail is contracted
// to fma(x1, x1, x0 * x0) on every x86-64 FMA3 build -- pinned by running the unmodified reference on 10^4 near-tie
// cases (tests/golden/icp_ties.npz; oracle/oracle.c: ref_norm2).  So the squared distance of the hot loop,
// fma(dy, dy, dx * dx), IS the reference's radicand bit for bit; what an argmin over it still misses is that sqrt
// merges neighbouring doubles: two candidates whose radicands differ in the last bits are a TIE for the reference
// (lowest j wins).  The search therefore works in two tiers:
//   * the hot loop compares only the HIGH 32 bits of the squared distance (non-negative doubles order like their
//     bit patterns; NaN patterns are above +inf and never win), which decides every pair of candidates that differ
//     by more than 2^-19 relative -- far outside anything a square root can merge -- and raises a flag whenever two
//     compared values are within one unit of that word (an integer subtract + min, no FP64 issue slot);
//   * a flagged source point (a few per 10^4) is re-done by the whole warp with the reference's own expression,
//     square root included: ref_dist / warp_careful_nearest.
__device__ __forceinline__ double ref_dist(double dx, double dy)
{
    return __dsqrt_rn(__fma_rn(dy, dy, __dmul_rn(dx, dx)));  // [ICP]:102
}

// Exhaustive search for ONE source point (px, py: warp-uniform) over all m targets by the reference's rule; the 32
// lanes take every 32nd target and the partial winners are merged with "smaller distance, then lower index".
// PAD_BLK > 0: the target array has one unused slot after every PAD_BLK points (queued search, see below).
template <int PAD_BLK>
static __device__ __noinline__ int warp_careful_nearest(double px, double py, const double2 *tar, int m, int lane)
{
    double bd = INFINITY;
    int bj = 0;
    for (int j = lane; j < m; j += 32) {
        const double2 t = tar[PAD_BLK ? j + j / PAD_BLK : j];
        const double d = ref_dist(px - t.x, py - t.y);
        if (d < bd) {
            bd = d;
            bj = j;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, bd, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        if (od < bd || (od == bd && oj < bj)) {
            bd = od;
            bj = oj;
        }
    }
    return bj;
}

// hi-word compare + near-tie flag of the hot loop
#define B2S_NN_STEP(FH, BH, BJ, J, NEAR)                    \
    do {                                                    \
        NEAR |= ((FH) - (BH) + 1u) < 3u;                    \
        if ((FH) < (BH)) {                                  \
            BH = (FH);                                      \
            BJ = (J);                                       \
        }                                                   \
    } while (0)

// ---------------------------------------------------------------- the queued search (PRUNE == 4, 5)
//
// The collective search (PRUNE 1..3) evaluates a block with the whole warp as soon as ONE of its 32 source points needs
// it: 32 consecutive points need the union of ~5 blocks, each point only 1-2 of them, so two thirds of the distance
// evaluations are spent on blocks the lane's own bound already excludes.  The queued search keeps the two pruning tests
// (same bounds, same proof) but only RECORDS what survives them: every (source point, block) pair that passes the
// per-lane test becomes one 4-byte item in a per-warp queue in shared memory, the items of a warp's R x 32 points are
// then spread evenly over the 32 lanes (lane l takes items l, l + 32, ...: one block of NN_BLK targets against one
// point each, so every evaluation is one some point needs), the per-item winners go to fixed result slots, and each
// point merges its own <= QK results in ascending block order with the same compare as everything else.  A point that
// needs more than QK blocks (a loose first-iteration bound, NaN coordinates) sends its whole group of 32 through the
// collective search instead.  For the items' loads to be conflict-free the target array carries one unused slot after
// every NN_BLK points (block stride NN_BLK + 1: neighbouring blocks start 4 banks apart), filled with NaN like the
// tail of a ragged last block -- NaN never wins and never raises the near-tie flag.
constexpr int QK = 3;                     // queued items (= result slots) per source point
constexpr int QCAND = 16;                 // candidate blocks of a group of 32 points beyond which it goes collective
constexpr int QSUP_MIN = 64;              // block count above which the warp test gets a second level (a bound per 32 blocks)
constexpr int QBLOCKS = 254;              // most blocks per target scan (block number + 1 fits a byte)

// Collective search of one group of 32 points on the padded target layout: the PRUNE == 2 algorithm (warp-level test,
// per-lane test, whole-warp visits).  Returns the winner's index, bit 31 = near-tie flag.
template <int NN_BLK>
static __device__ __noinline__ unsigned collective_nearest_padded(double px, double py, bool real, int arg_prev,
                                                                   const double2 *tar, const float4 *bnd, int nblk,
                                                                   int lane)
{
    const double2 g = tar[arg_prev + arg_prev / NN_BLK];
    const double gx = px - g.x, gy = py - g.y;
    const double ub = fma(gy, gy, gx * gx);
    const float suf = sqrt_up(__double2float_ru(ub));
    const float pxf = __double2float_rn(px), pyf = __double2float_rn(py);
    const float suE = __fmul_ru(__fadd_ru(suf, __fmul_ru(__fadd_ru(fabsf(pxf), fabsf(pyf)), 2.3841858e-7f)), 1.000002f);
    const int mid = __popc(__ballot_sync(0xffffffffu, real)) >> 1;
    const double wx = __shfl_sync(0xffffffffu, px, mid), wy = __shfl_sync(0xffffffffu, py, mid);
    const double ex = px - wx, ey = py - wy;
    const float ef = real ? __fadd_ru(sqrt_up(__double2float_ru(fma(ey, ey, ex * ex))), suf) * 1.000001f : 0.0f;
    const float gmax = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(ef)));
    const float wxf = __double2float_rn(wx), wyf = __double2float_rn(wy);
    const float gE = __fmul_ru(__fadd_ru(gmax, __fmul_ru(__fadd_ru(fabsf(wxf), fabsf(wyf)), 2.3841858e-7f)), 1.000002f);
    unsigned bh[NN_CHAINS];
    int bj[NN_CHAINS];
    bool near = false;
#pragma unroll
    for (int q = 0; q < NN_CHAINS; ++q) {
        bh[q] = 0x7ff00000u;
        bj[q] = 0;
    }
    for (int base = 0; base < nblk; base += 32) {
        bool keep = false;
        if (base + lane < nblk) {
            const float4 c = bnd[base + lane];
            const float cxd = wxf - c.x, cyd = wyf - c.y;
            const float reach = __fadd_ru(c.z, gE);
            keep = !(fmaf(cyd, cyd, cxd * cxd) > __fmul_ru(reach, reach));
        }
        unsigned todo = __ballot_sync(0xffffffffu, keep);
        while (todo) {
            const int b = base + __ffs(todo) - 1;
            todo &= todo - 1;
            const float4 c = bnd[b];
            const float cxd = pxf - c.x, cyd = pyf - c.y;
            const float reach = __fadd_ru(c.z, suE);
            const bool skip = !real || (fmaf(cyd, cyd, cxd * cxd) > __fmul_ru(reach, reach));
            if (__all_sync(0xffffffffu, skip)) continue;
            const double2 *blk = tar + b * (NN_BLK + 1);
#pragma unroll
            for (int jj = 0; jj < NN_BLK; ++jj) {
                const double2 t = blk[jj];
                const double dx = px - t.x, dy = py - t.y;
                const unsigned fh = (unsigned)__double2hiint(fma(dy, dy, dx * dx));
                B2S_NN_STEP(fh, bh[jj % NN_CHAINS], bj[jj % NN_CHAINS], b * NN_BLK + jj, near);
            }
        }
    }
#pragma unroll
    for (int q = 1; q < NN_CHAINS; ++q) B2S_NN_STEP(bh[q], bh[0], bj[0], bj[q], near);
    return (unsigned)bj[0] | (near ? 0x80000000u : 0u);
}

// Targets per pruning block (NN_BLK): 8 is fastest at 360 beams, 16 at 1080 with the warp-level test in front
// (16 / 32 with the per-lane test alone); chosen per launch, see launch_icp_r.

// Register cap: 80 per thread keeps 6 CTAs of 128 threads (360 beams) / 2 CTAs of 384 threads (1080 beams)
// resident per SM; without it the allocation of some instances drifts above that step from build to build.
// The small-scan instances (NN_BLK = 8, i.e. up to 600 targets: CTAs of 128 threads) fit 72 registers without a spill,
// which makes room for a 7th CTA per SM: measured 0.789 -> 0.765 ms on cfg 2; at 384 threads 72 registers buy no
// extra CTA and cost 1.4 %, and 64 registers (8 CTAs) spill 56 bytes and are slower than 72 on both shapes.
//
// RANGES = true is the fused-ingestion form (SURVEY 8f-1): tar_xy / src_xy hold raw ranges (one float per beam, n == m)
// and the points are formed here exactly as laserToNumpy does ([ICP]:216-229, [SLAM]:115-123): float64
// (cos a * r, sin a * r) with the beam table computed by the host's NumPy, +inf -> clamp when clamp > 0.
//
// ERR = true writes each pair's mean error of its last iteration ([ICP]:75) to err_out[pair].  It is a template
// parameter rather than a null test so that the instances without it compile to exactly the code they had before.
template <typename TIn, int R, int PRUNE, int NN_BLK, bool RANGES = false, bool ERR = false>
__global__ void __maxnreg__(R <= 3 ? (NN_BLK == 8 && PRUNE != 5 ? B2S_ICP_REGS_BLK8 : B2S_ICP_REGS_BLK16) : 104) icp_batch_kernel(const TIn *__restrict__ tar_xy, const TIn *__restrict__ src_xy, int n,
                                 int m, int max_iter, double tol, double *__restrict__ T_out,
                                 int32_t *__restrict__ iters_out, int use_bulk,
                                 const double2 *__restrict__ beam_cs = nullptr, double clamp = 0.0,
                                 double *__restrict__ err_out = nullptr)
{
    constexpr int ROWS = RANGES ? 1 : 2;  // values per point in the input arrays
    auto point = [&](const TIn *scan, int count, int i, double &x, double &y) {
        if (RANGES) {
            double r = (double)scan[i];
            if (clamp > 0.0 && r == INFINITY) r = clamp;  // [SLAM]:119 (only +inf compares equal)
            const double2 cs = beam_cs[i];
            x = __dmul_rn(cs.x, r);
            y = __dmul_rn(cs.y, r);
        } else {
            x = (double)scan[i];
            y = (double)scan[count + i];
        }
    };
    constexpr bool QUEUED = PRUNE >= 4;  // 5: with the second level of the warp test (a bound per 32 blocks)
    constexpr bool QSUP = PRUNE == 5;
    constexpr int PAD_BLK = QUEUED ? NN_BLK : 0;      // one unused slot after every PAD_BLK targets (queued search)
    // Per warp: QCAP queue entries (4 bytes) followed by QCAP result slots (8 bytes).
    constexpr int QCAP = R * QK * 32;
    static_assert(QK == 3, "phase C merges exactly three result slots");
    const int nblk = (m + NN_BLK - 1) / NN_BLK;
    auto TI = [](int j) { return PAD_BLK ? j + j / (PAD_BLK ? PAD_BLK : 1) : j; };  // index into tar[]
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // layout: [mbarrier 16 B][scratch][tar double2 * m (queued: nblk * (NN_BLK + 1))][staging TIn * 2m, 16-byte rounded]
    //         queued search only: [moved source double2 * R * threads][per warp: queue u32 * QCAP, results uint2 * QCAP]
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    double *scratch = reinterpret_cast<double *>(smem_raw + 16);
    double2 *tar = reinterpret_cast<double2 *>(smem_raw + 16 + icp_scratch_doubles(blockDim.x >> 5) * sizeof(double));
    const int tar_slots = QUEUED ? nblk * (NN_BLK + 1) : m;
    TIn *stage = reinterpret_cast<TIn *>(tar + tar_slots);
    double2 *srcm = reinterpret_cast<double2 *>(reinterpret_cast<unsigned char *>(stage) +
                                               icp_stage_bytes((size_t)ROWS * m * sizeof(TIn), nblk));
    unsigned *queue_all = reinterpret_cast<unsigned *>(srcm + (QUEUED ? R * blockDim.x : 0));  // 3 * QCAP words per warp

    const int pair = blockIdx.x;
    const int tid = threadIdx.x;
    const TIn *tar_g = tar_xy + (size_t)pair * ROWS * m;
    const TIn *src_g = src_xy + (size_t)pair * ROWS * n;

    // ---- stage the target scan: global -> shared via the bulk-copy engine when alignment allows
    if (use_bulk & 1) {
        if (tid == 0) {
            mbar_init(bar, 1);
            fence_mbar_init();
        }
        __syncthreads();
        if (tid == 0) {
            const uint32_t bytes = (uint32_t)ROWS * (uint32_t)m * (uint32_t)sizeof(TIn);
            mbar_expect_tx(bar, bytes);
            bulk_g2s(stage, tar_g, bytes, bar);
        }
    } else {
        for (int j = tid; j < ROWS * m; j += blockDim.x) stage[j] = tar_g[j];
    }

    // ---- this thread's source points (registers for the whole solve); overlaps the copy
    // The scan is cut into groups of `gs` consecutive points, the same number of groups for every warp (round r of warp
    // w holds group r * nwarps + w in its low lanes): 360 and 1080 beams both give groups of 30, so the warps reach the
    // one barrier of an iteration together instead of the last warp carrying a short tail group.
    const int nwarps_ = blockDim.x >> 5;
    const int rounds = ((n + 31) / 32 + nwarps_ - 1) / nwarps_;  // <= R by the launch geometry
    const int gs = (n + nwarps_ * rounds - 1) / (nwarps_ * rounds);
    // ... unless that takes more groups than the strided layout (point tid + r * threads, a short tail group), which
    // costs more than the imbalance (1080 beams on 12 warps: 36 against 34); use_bulk bits 1-2: 0 strided, 1 balanced, 2 auto
    const int layout = (use_bulk >> 1) & 3;
    const bool balanced = layout == 1 || (layout == 2 && nwarps_ * rounds <= (n + 31) / 32);
    auto point_index = [&](int r) -> int {  // -1: no point in this slot
        if (!balanced) return tid + r * (int)blockDim.x < n ? tid + r * (int)blockDim.x : -1;
        const int i = (r * nwarps_ + (tid >> 5)) * gs + (tid & 31);
        return (r < rounds && (tid & 31) < gs && i < n) ? i : -1;
    };
    double sx[R], sy[R];  // moved by every iteration; the originals are read again for the final fit
    int count = 0;
    double first[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = point_index(r);
        sx[r] = sy[r] = 0.0;
        if (i >= 0) {
            point(src_g, n, i, sx[r], sy[r]);
            count = r + 1;
            first[0] += sx[r];
            first[1] += sy[r];
        }
    }

    if (use_bulk & 1) mbar_wait(bar, 0);
    else __syncthreads();
    for (int j = tid; j < m; j += blockDim.x) {
        double2 t;
        point(stage, m, j, t.x, t.y);
        tar[TI(j)] = t;
        first[2] += t.x;
        first[3] += t.y;
    }
    if (QUEUED) {  // the unused slot of every block and the tail of a ragged last block: NaN never wins, never ties
        const double qnan = __longlong_as_double(0x7ff8000000000000LL);
        for (int b = tid; b < nblk; b += blockDim.x) tar[b * (NN_BLK + 1) + NN_BLK] = make_double2(qnan, qnan);
        for (int j = m + tid; j < nblk * NN_BLK; j += blockDim.x) tar[TI(j)] = make_double2(qnan, qnan);
    }
    // fixed shifts for the one-pass fits: centroid of the original source, centroid of the target scan
    block_sum<4>(first, scratch);  // its barriers also publish tar[]
    int phase = 0;
    // (any fixed value is a valid shift; a scan with NaN / inf points, which are never matched, falls back to 0)
    auto shift = [](double sum, int cnt) { const double c = sum / (double)cnt; return (fabs(c) < INFINITY) ? c : 0.0; };
    const double sax = shift(first[0], n), say = shift(first[1], n);
    const double sbx = shift(first[2], m), sby = shift(first[3], m);

    // ---- pruning bounds: the target scan is cut into blocks of NN_BLK consecutive points, each with a centre and a
    // radius that covers it.  The bounds only decide which blocks are LOOKED AT, never the result, so they live in
    // float32 (half the issue slots of the float64 tests they replace), made conservative as follows.  The centre is
    // the float32 rounding of the bounding-box centre -- any point serves as a centre as long as the radius is measured
    // from it, so the radius is taken in float64 from that float32 point and rounded UP.  A source point p enters the
    // test as pf = float(p), off by at most 2^-24 (|px| + |py|); the float32 distance computation adds at most 2^-22
    // relative.  A block is skipped iff  |pf - c|^2 (float)  >  ((rad + su + E) (1 + 2^-19))^2  rounded up, with
    // E = 2^-22 (|pfx| + |pfy|): then the true |p - c| exceeds rad + su, i.e. every point of the block is farther than
    // the upper bound su >= sqrt(ub) (1 + 2^-23) on the nearest distance.  NaN / inf anywhere make the comparison false:
    // nothing is skipped.  The staging area is free again and holds the bounds: [nblk] float4.
    float4 *bnd = reinterpret_cast<float4 *>(stage);
    if (PRUNE) {
        for (int b = tid; b < nblk; b += blockDim.x) {
            const int j0 = b * NN_BLK, j1 = min(m, j0 + NN_BLK);
            const double2 *tb = tar + TI(j0) - j0;  // (a block is contiguous in both layouts)
            double x0 = tb[j0].x, x1 = x0, y0 = tb[j0].y, y1 = y0;
            for (int j = j0 + 1; j < j1; ++j) {
                x0 = fmin(x0, tb[j].x); x1 = fmax(x1, tb[j].x);
                y0 = fmin(y0, tb[j].y); y1 = fmax(y1, tb[j].y);
            }
            const float cfx = __double2float_rn(0.5 * (x0 + x1)), cfy = __double2float_rn(0.5 * (y0 + y1));
            const double cx = (double)cfx, cy = (double)cfy;
            double rad2 = 0.0;
            bool finite = true;
            for (int j = j0; j < j1; ++j) {
                const double dx = tb[j].x - cx, dy = tb[j].y - cy;
                const double d2 = fma(dy, dy, dx * dx);
                finite = finite && (d2 == d2) && (d2 < INFINITY);
                rad2 = fmax(rad2, d2);
            }
            // a block with a NaN / inf point gets an infinite radius: it is never skipped
            const double rad = finite ? sqrt(rad2) * 1.000000001 + 1e-300 : INFINITY;
            bnd[b] = make_float4(cfx, cfy, __fmul_ru(__double2float_ru(rad), 1.000002f), 0.0f);  // (1 + 2^-19) folded in
        }
        __syncthreads();
        if (QSUP) {
            // one more level for the warp test: a circle around every 32 consecutive blocks (centre: the float32 centre of
            // their centres' bounding box, radius: farthest block centre + that block's radius, rounded up), so that a warp
            // looks only at the groups of 32 blocks it can reach.  Same argument, same margins as for a block.
            float4 *sup = bnd + nblk;
            const int lane_ = tid & 31;
            for (int g = tid >> 5; g < (nblk + 31) / 32; g += (int)(blockDim.x >> 5)) {  // one warp per group, one block per lane
                const int b = min(nblk - 1, g * 32 + lane_);  // (the tail lanes repeat the last block)
                const float4 c = bnd[b];
                float x0 = c.x, x1 = c.x, y0 = c.y, y1 = c.y;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    x0 = fminf(x0, __shfl_xor_sync(0xffffffffu, x0, o)); x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, o));
                    y0 = fminf(y0, __shfl_xor_sync(0xffffffffu, y0, o)); y1 = fmaxf(y1, __shfl_xor_sync(0xffffffffu, y1, o));
                }
                const float cfx = 0.5f * x0 + 0.5f * x1, cfy = 0.5f * y0 + 0.5f * y1;  // (any point serves as a centre)
                const double dx = (double)c.x - (double)cfx, dy = (double)c.y - (double)cfy;
                const double d = sqrt(fma(dy, dy, dx * dx)) * 1.000000001 + (double)c.z;
                // rounded up to float32; NaN / inf (a block that is never skipped, a non-finite centre) order above all
                // finite values as unsigned bit patterns of non-negative floats, so one REDUX takes the maximum
                float df = __fmul_ru(__double2float_ru(d), 1.000002f);
                if (!(df >= 0.0f) || !(fabsf(cfx) < INFINITY) || !(fabsf(cfy) < INFINITY)) df = INFINITY;
                const float reach = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(df)));
                if (lane_ == 0)
                    sup[g] = make_float4(reach < INFINITY ? cfx : 0.0f, reach < INFINITY ? cfy : 0.0f, reach, 0.0f);
            }
            __syncthreads();
        }
    }

    // previous match of every source point; seeds the pruning bound (first pass: the target with the
    // proportional index, which is the same beam when both scans have the same beam count)
    int arg[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const long long i = max(0, point_index(r));
        arg[r] = (int)min((long long)(m - 1), i * m / n);
    }

    if (QUEUED) {
#pragma unroll
        for (int r = 0; r < R; ++r) srcm[tid + r * blockDim.x] = make_double2(sx[r], sy[r]);
    }

    double prev_err = 0.0, err = 0.0;  // err after the loop: the mean error of the last iteration run
    int iters = 0;
    for (int it = 0; it < max_iter; ++it) {
        // ---- nearest neighbour ([ICP]:99-106)
        const int lane_id = tid & 31;
        // re-do flagged points (near ties: see ref_dist) with the reference's expression; warp-uniform
        auto settle = [&](bool flagged, double px, double py, int &winner) {
            unsigned need = __ballot_sync(0xffffffffu, flagged);
            while (need) {
                const int src_lane = __ffs(need) - 1;
                need &= need - 1;
                const double qx = __shfl_sync(0xffffffffu, px, src_lane), qy = __shfl_sync(0xffffffffu, py, src_lane);
                const int j = warp_careful_nearest<PAD_BLK>(qx, qy, tar, m, lane_id);
                if (lane_id == src_lane) winner = j;
            }
        };
        if (!PRUNE) {
            unsigned bh[R];
            bool near[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                bh[r] = 0x7ff00000u;  // +inf
                arg[r] = 0;
                near[r] = false;
            }
#pragma unroll 4
            for (int j = 0; j < m; ++j) {
                const double2 t = tar[j];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const double dx = sx[r] - t.x, dy = sy[r] - t.y;
                    const unsigned fh = (unsigned)__double2hiint(fma(dy, dy, dx * dx));
                    B2S_NN_STEP(fh, bh[r], arg[r], j, near[r]);
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) settle(near[r] && r < count, sx[r], sy[r], arg[r]);
        } else if (QUEUED) {
            const int lane = tid & 31;
            unsigned *q = queue_all + (tid >> 5) * (3 * QCAP);
            uint2 *res = reinterpret_cast<uint2 *>(q + QCAP);
            const unsigned lt = (1u << lane) - 1u;
            unsigned total = 0;       // items queued by this warp (warp-uniform)
            unsigned collective = 0;  // bit r: group r goes through the collective search
            int cnt[R];
            // ---- phase A: the two pruning tests; what survives is queued, one candidate block after the other
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const bool real = r < count;
                const double px = sx[r], py = sy[r];
                const double2 g = tar[TI(arg[r])];
                const double gx = px - g.x, gy = py - g.y;
                const double ub = fma(gy, gy, gx * gx);
                const float suf = sqrt_up(__double2float_ru(ub));
                const float pxf = __double2float_rn(px), pyf = __double2float_rn(py);
                const float suE = __fmul_ru(__fadd_ru(suf, __fmul_ru(__fadd_ru(fabsf(pxf), fabsf(pyf)), 2.3841858e-7f)),
                                            1.000002f);
                const int mid = __popc(__ballot_sync(0xffffffffu, real)) >> 1;
                const double wx = __shfl_sync(0xffffffffu, px, mid), wy = __shfl_sync(0xffffffffu, py, mid);
                const double ex = px - wx, ey = py - wy;
                const float ef = real ? __fadd_ru(sqrt_up(__double2float_ru(fma(ey, ey, ex * ex))), suf) * 1.000001f
                                      : 0.0f;
                const float gmax = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(ef)));
                const float wxf = __double2float_rn(wx), wyf = __double2float_rn(wy);
                const float gE = __fmul_ru(__fadd_ru(gmax, __fmul_ru(__fadd_ru(fabsf(wxf), fabsf(wyf)), 2.3841858e-7f)),
                                           1.000002f);
                // item: point slot (12 bits) | block (10 bits) << 12 | result slot r * QK + k (4 bits) << 22
                const unsigned item0 = (unsigned)(tid + r * blockDim.x) | ((unsigned)(r * QK) << 22);
                unsigned mine = 0;  // byte k: 1 + the k-th block this point needs (ascending)
                unsigned sh = 0;    // 8 x the number of blocks it needs (shl_sat drops what does not fit)
                int ncand = 0;
                unsigned groups = 0xffffffffu >> (32 - (nblk + 31) / 32);  // bit g: blocks 32 g .. 32 g + 31
                if (QSUP) {  // (a template parameter: with two groups or fewer the extra level costs more than it saves)
                    bool far = false;
                    if (lane < (nblk + 31) / 32) {  // lane g: can the warp reach any block of group g ?
                        const float4 cs = bnd[nblk + lane];
                        const float cxd = wxf - cs.x, cyd = wyf - cs.y;
                        const float reach = __fadd_ru(cs.z, gE);
                        far = fmaf(cyd, cyd, cxd * cxd) > __fmul_ru(reach, reach);
                    }
                    groups &= ~__ballot_sync(0xffffffffu, far);
                }
                while (groups) {
                    const int base = (__ffs(groups) - 1) * 32;
                    groups &= groups - 1;
                    bool keep = false;
                    if (base + lane < nblk) {
                        const float4 cb = bnd[base + lane];
                        const float cxd = wxf - cb.x, cyd = wyf - cb.y;
                        const float reach = __fadd_ru(cb.z, gE);
                        keep = !(fmaf(cyd, cyd, cxd * cxd) > __fmul_ru(reach, reach));
                    }
                    unsigned todo = __ballot_sync(0xffffffffu, keep);
                    ncand += __popc(todo);
                    if (ncand > QCAND) break;  // a bound this loose: the collective search wastes less
                    while (todo) {  // two candidate blocks per pass (independent loads and tests)
                        const int b0 = base + __ffs(todo) - 1;
                        todo &= todo - 1;
                        const bool two = todo != 0;
                        const int b1 = two ? base + __ffs(todo) - 1 : b0;
                        todo &= todo - 1;
                        const float4 c0 = bnd[b0], c1 = bnd[b1];
                        const float x0 = pxf - c0.x, y0 = pyf - c0.y, x1 = pxf - c1.x, y1 = pyf - c1.y;
                        const float reach0 = __fadd_ru(c0.z, suE), reach1 = __fadd_ru(c1.z, suE);
                        const bool need0 = real && !(fmaf(y0, y0, x0 * x0) > __fmul_ru(reach0, reach0));
                        const bool need1 = real && two && !(fmaf(y1, y1, x1 * x1) > __fmul_ru(reach1, reach1));
                        if (need0) {
                            mine |= shl_sat((unsigned)b0 + 1u, sh);
                            sh += 8;
                        }
                        if (need1) {
                            mine |= shl_sat((unsigned)b1 + 1u, sh);
                            sh += 8;
                        }
                    }
                }
                const int c = (int)(sh >> 3);
                // too many candidate blocks, or a point that needs more blocks than it has result slots
                if (ncand > QCAND || __any_sync(0xffffffffu, c > QK)) {
                    collective |= 1u << r;
                } else {
                    static_assert(QK <= 3, "the two ballots below count up to 3 items per point");
                    const unsigned c0 = __ballot_sync(0xffffffffu, (c & 1) != 0), c1 = __ballot_sync(0xffffffffu, (c & 2) != 0);
                    const unsigned at = total + __popc(c0 & lt) + 2 * __popc(c1 & lt);
#pragma unroll
                    for (int k = 0; k < QK; ++k)
                        if (k < c) q[at + k] = item0 + ((((mine >> (8 * k)) & 255u) - 1u) << 12) + ((unsigned)k << 22);
                    total += __popc(c0) + 2 * __popc(c1);
                }
                cnt[r] = c;
            }
            __syncwarp();
            // ---- phase B: one item per lane and pass, NN_BLK targets against one point.  The block-local index rides in
            // the low bits of the key (high word of the squared distance, low bits masked), so the smallest and the
            // second smallest key of the block come out of a min / max tournament; two keys less than two mask units
            // apart raise the near-tie flag (the exhaustive careful search then decides).
            constexpr unsigned KMASK = NN_BLK - 1;  // NN_BLK is a power of two
            for (unsigned t0 = 0; t0 < total; t0 += 32) {
                const unsigned t = t0 + lane;
                const bool valid = t < total;
                const unsigned e = q[valid ? t : 0u];  // (an idle lane repeats item 0 and drops the result)
                const double2 p = srcm[e & 0xfffu];
                const unsigned b = (e >> 12) & 0x3ffu;
                const double2 *blk = tar + b * (NN_BLK + 1);
                unsigned lo[NN_BLK], hi[NN_BLK];
#pragma unroll
                for (int jj = 0; jj < NN_BLK; ++jj) {
                    const double2 tg = blk[jj];
                    const double dx = p.x - tg.x, dy = p.y - tg.y;
                    lo[jj] = ((unsigned)__double2hiint(fma(dy, dy, dx * dx)) & ~KMASK) | (unsigned)jj;
                }
#pragma unroll
                for (int jj = 0; jj < NN_BLK; jj += 2) {
                    const unsigned x = lo[jj], y = lo[jj + 1];
                    lo[jj] = min(x, y);
                    hi[jj] = max(x, y);
                }
#pragma unroll
                for (int w = 2; w < NN_BLK; w *= 2)
#pragma unroll
                    for (int jj = 0; jj < NN_BLK; jj += 2 * w) {
                        const unsigned la = lo[jj], lb = lo[jj + w];
                        hi[jj] = min(min(hi[jj], hi[jj + w]), max(la, lb));
                        lo[jj] = min(la, lb);
                    }
                const bool near = ((hi[0] & ~KMASK) - (lo[0] & ~KMASK)) <= NN_BLK;
                if (valid) res[(e >> 22) * 32 + (e & 31u)] = make_uint2(lo[0], b | (near ? 0x80000000u : 0u));
            }
            __syncwarp();
            // ---- phase C: every point merges its own (up to QK) results; branch-free, the two smallest masked keys
            // decide the near-tie flag exactly as inside a block
            unsigned flagged = 0;  // bit r: point r of this lane is a near tie
#pragma unroll
            for (int r = 0; r < R; ++r) {
                bool near = false;
                if (collective & (1u << r)) {
                    const unsigned w = collective_nearest_padded<NN_BLK>(sx[r], sy[r], r < count, arg[r], tar, bnd, nblk, lane);
                    arg[r] = (int)(w & 0x7fffffffu);
                    near = (w >> 31) != 0;
                } else {
                    const int c = cnt[r];
                    uint2 v[QK];
                    unsigned f[QK];
#pragma unroll
                    for (int k = 0; k < QK; ++k) {
                        v[k] = res[(r * QK + k) * 32 + lane];
                        f[k] = k < c ? (v[k].x & ~KMASK) : 0xffffffffu;
                        near |= k < c && (v[k].y >> 31) != 0;
                    }
                    const unsigned best = min(f[0], min(f[1], f[2]));
                    const unsigned second = max(min(f[0], f[1]), min(max(f[0], f[1]), f[2]));  // median of three
                    const uint2 win = f[0] == best ? v[0] : (f[1] == best ? v[1] : v[2]);
                    arg[r] = c ? (int)((win.y & 0x3ffu) * NN_BLK + (win.x & KMASK)) : 0;
                    // two blocks' minima less than two mask units apart, or nothing finite at all: the careful search decides
                    near |= c && (second - best <= (unsigned)NN_BLK || best >= 0x7ff00000u);
                }
                flagged |= (near && r < count) ? (1u << r) : 0u;
            }
            if (__any_sync(0xffffffffu, flagged != 0)) {
#pragma unroll
                for (int r = 0; r < R; ++r) settle((flagged >> r) & 1u, sx[r], sy[r], arg[r]);
            }
        } else {
            // Exact search with pruning.  ANY target gives an upper bound ub on the nearest distance; a block
            // whose every point is provably farther than sqrt(ub) cannot contain the nearest point nor tie
            // with it, so it is skipped.  Blocks are visited in ascending order and their points compared
            // with the same strict '<', so the winner (lowest index among equals) is the brute-force one.
            // The 32 lanes of a warp hold 32 consecutive source points for a given r, so they agree on almost
            // all blocks; a block is evaluated by the whole warp as soon as one lane needs it.
            //
            // PRUNE == 2 puts a warp-level test in front: the 32 source points of the warp lie within g of a
            // common centre w (g = max over lanes of |p - w| + sqrt(ub), rounded UP to float and reduced with one
            // REDUX), so a block whose centre is farther than radius + g from w is skipped for every lane by the
            // triangle inequality.  Lane b tests block b, i.e. 32 blocks per instruction sequence instead of one,
            // and only the surviving few blocks reach the per-lane test.  NaN / inf anywhere makes the comparison
            // false, i.e. nothing is skipped.
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const bool real = r < count;
                const double px = sx[r], py = sy[r];
                const double2 g = tar[TI(arg[r])];
                const double gx = px - g.x, gy = py - g.y;
                const double ub = fma(gy, gy, gx * gx);
                // sqrt(ub) rounded UP in float (two instructions instead of a double-precision square root); an
                // upper bound is all the tests need.  NaN stays NaN, overflow gives inf: then nothing is skipped.
                // The factor (> 1 + 2^-23) covers the rounding of the double-precision tests below.
                const float suf = sqrt_up(__double2float_ru(ub));
                // the point in float32 for the block tests, its rounding allowance E, and su + E with the (1 + 2^-19)
                const float pxf = __double2float_rn(px), pyf = __double2float_rn(py);
                const float suE = __fmul_ru(__fadd_ru(suf, __fmul_ru(__fadd_ru(fabsf(pxf), fabsf(pyf)), 2.3841858e-7f)),
                                            1.000002f);
                // NN_CHAINS independent running minima (target j feeds chain j % NN_CHAINS) shorten the serial
                // compare-select dependency; they are merged below with the lower index winning ties, which is
                // what one ascending strict '<' scan gives.
                unsigned bh[NN_CHAINS];  // high word of the chain's smallest squared distance
                int bj[NN_CHAINS];
                bool near = false;
#pragma unroll
                for (int q = 0; q < NN_CHAINS; ++q) {
                    bh[q] = 0x7ff00000u;  // +inf
                    bj[q] = 0;
                }
                auto visit = [&](int b) {
                    const int j0 = b * NN_BLK;
                    if (j0 + NN_BLK <= m) {
#pragma unroll
                        for (int jj = 0; jj < NN_BLK; ++jj) {
                            const double2 t = tar[j0 + jj];
                            const double dx = px - t.x, dy = py - t.y;
                            const unsigned fh = (unsigned)__double2hiint(fma(dy, dy, dx * dx));
                            B2S_NN_STEP(fh, bh[jj % NN_CHAINS], bj[jj % NN_CHAINS], j0 + jj, near);
                        }
                    } else {
                        for (int j = j0; j < m; ++j) {
                            const double2 t = tar[j];
                            const double dx = px - t.x, dy = py - t.y;
                            const unsigned fh = (unsigned)__double2hiint(fma(dy, dy, dx * dx));
                            B2S_NN_STEP(fh, bh[0], bj[0], j, near);  // (the ragged block is the last one: still ascending)
                        }
                    }
                };
                auto lane_skips = [&](int b) -> bool {
                    const float4 c = bnd[b];
                    const float cxd = pxf - c.x, cyd = pyf - c.y;
                    const float dc2 = fmaf(cyd, cyd, cxd * cxd);
                    const float reach = __fadd_ru(c.z, suE);
                    return !real || (dc2 > __fmul_ru(reach, reach));
                };
                if (PRUNE >= 2) {
                    // common centre: the middle lane's point (any point works; the bound is computed from the actual points)
                    const int mid = __popc(__ballot_sync(0xffffffffu, real)) >> 1;  // real lanes are the low ones
                    const double wx = __shfl_sync(0xffffffffu, px, mid), wy = __shfl_sync(0xffffffffu, py, mid);
                    const double ex = px - wx, ey = py - wy;
                    const float ef = real ? __fadd_ru(sqrt_up(__double2float_ru(fma(ey, ey, ex * ex))), suf) * 1.000001f
                                          : 0.0f;  // every step rounds up; NaN bits compare above all
                    const float gmax = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(ef)));
                    // the same float32 test as lane_skips, for the common centre w and the warp's bound gmax
                    const float wxf = __double2float_rn(wx), wyf = __double2float_rn(wy);
                    const float gE = __fmul_ru(__fadd_ru(gmax, __fmul_ru(__fadd_ru(fabsf(wxf), fabsf(wyf)), 2.3841858e-7f)),
                                               1.000002f);
                    const int lane = tid & 31;
                    for (int base = 0; base < nblk; base += 32) {
                        bool keep = false;
                        if (base + lane < nblk) {
                            const float4 c = bnd[base + lane];
                            const float cxd = wxf - c.x, cyd = wyf - c.y;
                            const float dc2 = fmaf(cyd, cyd, cxd * cxd);
                            const float reach = __fadd_ru(c.z, gE);
                            keep = !(dc2 > __fmul_ru(reach, reach));
                        }
                        unsigned todo = __ballot_sync(0xffffffffu, keep);
                        while (todo) {
                            const int b = base + __ffs(todo) - 1;
                            todo &= todo - 1;
                            if (PRUNE == 2 && __all_sync(0xffffffffu, lane_skips(b))) continue;  // PRUNE 3: warp test only
                            visit(b);
                        }
                    }
                } else {
                    for (int b = 0; b < nblk; ++b) {
                        if (__all_sync(0xffffffffu, lane_skips(b))) continue;
                        visit(b);
                    }
                }
#pragma unroll
                for (int q = 1; q < NN_CHAINS; ++q) B2S_NN_STEP(bh[q], bh[0], bj[0], bj[q], near);
                arg[r] = bj[0];
                settle(near && real, px, py, arg[r]);
            }
        }
        // ---- matched targets, distances ([ICP]:69,75)
        double bx[R], by[R];
        double dsum = 0.0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (PRUNE && r >= count) arg[r] = 0;  // idle slot: keep the index in range
            const double2 t = tar[TI(arg[r])];
            bx[r] = t.x;
            by[r] = t.y;
            if (r < count) {
                const double d = ref_dist(sx[r] - t.x, sy[r] - t.y);  // [ICP]:102; inf / NaN: nothing was matched,
                dsum += (d < INFINITY) ? d : 0.0;                     // the reference keeps distance 0 ([ICP]:95)
            }
        }
        double T[6];
        cta_rigid_fit<R>(sx, sy, bx, by, count, n, sax, say, sbx, sby, dsum, scratch, phase, T);
        // ---- src <- T . src ([ICP]:71)
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const double x = sx[r], y = sy[r];
            sx[r] = T[0] * x + T[1] * y + T[2];
            sy[r] = T[3] * x + T[4] * y + T[5];
            if (QUEUED) srcm[tid + r * blockDim.x] = make_double2(sx[r], sy[r]);
        }
        ++iters;
        err = dsum / (double)n;
        if (fabs(prev_err - err) < tol) break;  // [ICP]:76, uniform across the CTA
        prev_err = err;
    }

    if (ERR && tid == 0) err_out[pair] = err;  // (here rather than below: err is not held across the final fit)
    double T[6];
    double unused = 0.0;
    double ox_[R], oy_[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = point_index(r);
        ox_[r] = oy_[r] = 0.0;
        if (i >= 0) point(src_g, n, i, ox_[r], oy_[r]);
    }
    cta_rigid_fit<R>(ox_, oy_, sx, sy, count, n, sax, say, sax, say, unused, scratch, phase, T);  // [ICP]:81
    if (tid == 0) {
        double *o = T_out + (size_t)pair * 9;
        o[0] = T[0]; o[1] = T[1]; o[2] = T[2];
        o[3] = T[3]; o[4] = T[4]; o[5] = T[5];
        o[6] = 0.0;  o[7] = 0.0;  o[8] = 1.0;
        if (iters_out) iters_out[pair] = iters;
    }
}

extern int g_icp_src_per_thread;
extern int g_icp_prune;
extern int g_icp_block;
extern int g_icp_layout;

// Dynamic shared memory of one CTA (the layout at the top of the kernel); in_bytes = bytes of the staged input rows.
template <int PRUNE, int NN_BLK, int R>
static size_t icp_smem_bytes(int n_tar, size_t in_bytes, int threads)
{
    const size_t nblk = ((size_t)n_tar + NN_BLK - 1) / NN_BLK;
    size_t bytes = 16 + icp_scratch_doubles(threads / 32) * sizeof(double) + icp_stage_bytes(in_bytes, (int)nblk);
    if (PRUNE >= 4) {
        bytes += nblk * (NN_BLK + 1) * sizeof(double2);                       // padded targets
        bytes += (size_t)R * threads * sizeof(double2);                       // moved source points
        bytes += (size_t)(threads / 32) * (size_t)(R * QK * 32) * (sizeof(unsigned) + sizeof(uint2));  // queues + results
    } else {
        bytes += (size_t)n_tar * sizeof(double2);
    }
    return bytes;
}

template <typename TIn, int R, int PRUNE, int NN_BLK>
static int launch_icp_rp(const TIn *tar_xy, const TIn *src_xy, int pairs, int n_src, int n_tar, int max_iter,
                        double tol, double *T_out, int32_t *iters_out, double *err_out, void *stream)
{
    int threads = (n_src + R - 1) / R;
    threads = ((threads + 31) / 32) * 32;
    if (threads < 64) threads = 64;
    B2S_REQUIRE(threads <= 1024, "b2s_icp_batch: too many source points per scan");
    const size_t smem = icp_smem_bytes<PRUNE, NN_BLK, R>(n_tar, (size_t)n_tar * 2 * sizeof(TIn), threads);
    B2S_REQUIRE(smem <= 227 * 1024, "b2s_icp_batch: n_tar too large for shared memory");
    // the score output exists for float64 clouds only (the relocalization's virtual scans and laserToNumpy points)
    constexpr bool HAS_ERR = sizeof(TIn) == 8;
    auto kernel = icp_batch_kernel<TIn, R, PRUNE, NN_BLK>;
    if (HAS_ERR && err_out) kernel = icp_batch_kernel<TIn, R, PRUNE, NN_BLK, false, HAS_ERR>;
    // opt-in above 48 KB; the attribute is per device and per function, and setting it is cheap
    if (smem > 48 * 1024)
        B2S_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // bulk copy needs 16-byte aligned source and size: every pair's target block must qualify
    const size_t pair_bytes = (size_t)2 * n_tar * sizeof(TIn);
    const int use_bulk = (((uintptr_t)tar_xy % 16 == 0) && (pair_bytes % 16 == 0) ? 1 : 0) | (g_icp_layout << 1);
    if (threads > 512) {  // (large scans only: the query is not free)
        cudaFuncAttributes fa;
        B2S_CUDA(cudaFuncGetAttributes(&fa, kernel));
        B2S_REQUIRE(threads <= fa.maxThreadsPerBlock, "b2s_icp_batch: scan too large for one CTA's registers");
    }
    kernel<<<pairs, threads, smem, (cudaStream_t)stream>>>(
        tar_xy, src_xy, n_src, n_tar, max_iter, tol, T_out, iters_out, use_bulk, nullptr, 0.0, err_out);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

template <typename TIn, int R>
static int launch_icp_r(const TIn *tar_xy, const TIn *src_xy, int pairs, int n_src, int n_tar, int max_iter,
                        double tol, double *T_out, int32_t *iters_out, double *err_out, void *stream)
{
    // the block bounds live in the staging area: [ceil(m/blk)] float4 must fit in 2*m*sizeof(TIn)
    const int blk = (g_icp_block == 8 || g_icp_block == 16 || g_icp_block == 32) ? g_icp_block
                    : (g_icp_prune == 4 ? 8 : g_icp_prune >= 2 ? (n_tar <= 600 ? 8 : 16) : (n_tar <= 600 ? 16 : 32));  // measured best per mode
    const bool fits = (size_t)((n_tar + blk - 1) / blk) * 16 <= (size_t)2 * n_tar * sizeof(TIn);
#define B2S_ICP_GO(P, B) \
    return launch_icp_rp<TIn, R, P, B>(tar_xy, src_xy, pairs, n_src, n_tar, max_iter, tol, T_out, iters_out, err_out, stream)
    if (g_icp_prune && fits) {
        if (g_icp_prune == 4) {  // (block numbers travel in one byte; beyond that the collective search takes over)
            if (blk == 8 && (n_tar + 7) / 8 <= QBLOCKS) {
                if ((n_tar + 7) / 8 > QSUP_MIN) B2S_ICP_GO(5, 8);
                B2S_ICP_GO(4, 8);
            }
            if ((n_tar + 15) / 16 <= QBLOCKS) {
                if ((n_tar + 15) / 16 > QSUP_MIN) B2S_ICP_GO(5, 16);
                B2S_ICP_GO(4, 16);
            }
        }
        if (g_icp_prune == 3) {
            if (blk == 8) B2S_ICP_GO(3, 8);
            if (blk == 16) B2S_ICP_GO(3, 16);
            B2S_ICP_GO(3, 32);
        }
        if (g_icp_prune == 2 || g_icp_prune == 4) {
            if (blk == 8) B2S_ICP_GO(2, 8);
            if (blk == 16) B2S_ICP_GO(2, 16);
            B2S_ICP_GO(2, 32);
        }
        if (blk == 8) B2S_ICP_GO(1, 16);
        if (blk == 16) B2S_ICP_GO(1, 16);
        B2S_ICP_GO(1, 32);
    }
    B2S_ICP_GO(0, 16);
#undef B2S_ICP_GO
}

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

// Fused-ingestion form: raw ranges + beam table (always the default search, PRUNE = 2).
template <int R, int NN_BLK, int PRUNE>
static int launch_icp_ranges_rbp(const float *tar_r, const float *src_r, const double *beam_cs, double clamp, int pairs,
                                int n, int max_iter, double tol, double *T_out, int32_t *iters_out, void *stream)
{
    int threads = ((((n + R - 1) / R) + 31) / 32) * 32;
    if (threads < 64) threads = 64;
    B2S_REQUIRE(threads <= 1024, "b2s_icp_batch_ranges: too many beams per scan");
    const size_t smem = icp_smem_bytes<PRUNE, NN_BLK, R>(n, (size_t)n * sizeof(float), threads);
    B2S_REQUIRE(smem <= 227 * 1024, "b2s_icp_batch_ranges: too many beams for shared memory");
    if (smem > 48 * 1024)
        B2S_CUDA(cudaFuncSetAttribute(icp_batch_kernel<float, R, PRUNE, NN_BLK, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
    if (threads > 512) {  // (large scans only: the query is not free)
        cudaFuncAttributes fa;
        B2S_CUDA(cudaFuncGetAttributes(&fa, icp_batch_kernel<float, R, PRUNE, NN_BLK, true>));
        B2S_REQUIRE(threads <= fa.maxThreadsPerBlock, "b2s_icp_batch_ranges: scan too large for one CTA's registers");
    }
    const int use_bulk = (((uintptr_t)tar_r % 16 == 0) && (((size_t)n * sizeof(float)) % 16 == 0) ? 1 : 0) | (g_icp_layout << 1);
    icp_batch_kernel<float, R, PRUNE, NN_BLK, true><<<pairs, threads, smem, (cudaStream_t)stream>>>(
        tar_r, src_r, n, n, max_iter, tol, T_out, iters_out, use_bulk, reinterpret_cast<const double2 *>(beam_cs), clamp);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

template <int R>
static int launch_icp_ranges_r(const float *tar_r, const float *src_r, const double *beam_cs, double clamp, int pairs,
                               int n, int max_iter, double tol, double *T_out, int32_t *iters_out, void *stream)
{
    // (the fused-ingestion form has the two default searches: queued, and the collective one of icp_prune 0..3)
    const int blk = (g_icp_block == 8 || g_icp_block == 16 || g_icp_block == 32) ? g_icp_block : (g_icp_prune == 4 || n <= 600 ? 8 : 16);
#define B2S_ICP_GO(B, P) \
    return launch_icp_ranges_rbp<R, B, P>(tar_r, src_r, beam_cs, clamp, pairs, n, max_iter, tol, T_out, iters_out, stream)
    if (g_icp_prune == 4) {
        if (blk == 8 && (n + 7) / 8 <= QBLOCKS) {
            if ((n + 7) / 8 > QSUP_MIN) B2S_ICP_GO(8, 5);
            B2S_ICP_GO(8, 4);
        }
        if ((n + 15) / 16 <= QBLOCKS) {
            if ((n + 15) / 16 > QSUP_MIN) B2S_ICP_GO(16, 5);
            B2S_ICP_GO(16, 4);
        }
    }
    if (blk == 8) B2S_ICP_GO(8, 2);
    if (blk == 16) B2S_ICP_GO(16, 2);
    B2S_ICP_GO(32, 2);
#undef B2S_ICP_GO
}

static int launch_icp_ranges(const float *tar_r, const float *src_r, const double *beam_cs, double clamp, int pairs, int n,
                             int max_iter, double tol, double *T_out, int32_t *iters_out, void *stream)
{
    B2S_REQUIRE(pairs >= 0 && n > 0 && max_iter >= 0, "b2s_icp_batch_ranges: bad sizes");
    if (pairs == 0) return B2S_OK;
    B2S_REQUIRE(tar_r && src_r && beam_cs && T_out, "b2s_icp_batch_ranges: null pointer");
    B2S_REQUIRE((uintptr_t)beam_cs % 16 == 0, "b2s_icp_batch_ranges: the beam table must be 16-byte aligned");
    B2S_REQUIRE(tol == tol && clamp == clamp, "b2s_icp_batch_ranges: NaN tolerance / clamp");
    B2S_REQUIRE(n <= ICP_MAX_POINTS, "b2s_icp_batch_ranges: more than 2304 beams per scan is not supported");
    switch (icp_points_per_thread(n)) {
    case 2: return launch_icp_ranges_r<2>(tar_r, src_r, beam_cs, clamp, pairs, n, max_iter, tol, T_out, iters_out, stream);
    case 3: return launch_icp_ranges_r<3>(tar_r, src_r, beam_cs, clamp, pairs, n, max_iter, tol, T_out, iters_out, stream);
    default: return launch_icp_ranges_r<4>(tar_r, src_r, beam_cs, clamp, pairs, n, max_iter, tol, T_out, iters_out, stream);
    }
}

// err_out [pairs] (may be NULL): the reference's mean_error ([ICP]:75) of each pair's last iteration.
template <typename TIn>
static int launch_icp(const TIn *tar_xy, const TIn *src_xy, int pairs, int n_src, int n_tar,
                      int max_iter, double tol, double *T_out, int32_t *iters_out, double *err_out, void *stream)
{
    B2S_REQUIRE(pairs >= 0 && n_src > 0 && n_tar > 0 && max_iter >= 0, "b2s_icp_batch: bad sizes");
    if (pairs == 0) return B2S_OK;
    B2S_REQUIRE(tar_xy && src_xy && T_out, "b2s_icp_batch: null pointer");
    B2S_REQUIRE(tol == tol, "b2s_icp_batch: NaN tolerance");
    B2S_REQUIRE(n_src <= ICP_MAX_POINTS, "b2s_icp_batch: more than 2304 source points per scan is not supported");
    const int r = icp_points_per_thread(n_src);
    switch (r) {
    case 2: return launch_icp_r<TIn, 2>(tar_xy, src_xy, pairs, n_src, n_tar, max_iter, tol, T_out, iters_out, err_out, stream);
    case 3: return launch_icp_r<TIn, 3>(tar_xy, src_xy, pairs, n_src, n_tar, max_iter, tol, T_out, iters_out, err_out, stream);
    default: return launch_icp_r<TIn, 4>(tar_xy, src_xy, pairs, n_src, n_tar, max_iter, tol, T_out, iters_out, err_out, stream);
    }
}

}  // namespace b2s
