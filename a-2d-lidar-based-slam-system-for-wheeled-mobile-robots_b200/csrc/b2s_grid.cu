// Occupancy-grid kernels: Bresenham ray-cast into int32 hit/miss planes, finalize, ROS packing.
//
// Replaces Mapping.update ([MAP]:22-51) with bresenham ([BRES]:2-58) inlined.  Cell indices are
// bit-exact against the reference: the world->cell transform and the Bresenham error term are
// evaluated in float64 with the reference's operation order, one sequential recurrence per beam.
//
// Layout in HBM: hit, miss int32 [xw][yw] x-major (reference datamap[x][y]); endpoints ox, oy
// float32 [scans][beams] (SoA, as the reference passes two arrays); sensor positions cx, cy
// float32 [scans].  One lane per beam, so a warp reads 32 consecutive endpoints (coalesced) and
// its 32 rays fan out from the same sensor cell.
#include "b2s_common.cuh"

namespace b2s {

// 1: one RED per visit; 2: warp-aggregated runs; 3: same, lean inner loop;
// 4: 3 + transposed scratch plane for y-major beams when a workspace is supplied, else 3;
// 5: 4 + a test-free core phase of the march; 6 (default): consecutive scans counted in a shared-memory tile, 5 where
// the tile does not fit
int g_grid_variant = 6;

// ------------------------------------------------------------------------------------------
// Per-beam setup shared by all variants.

struct Beam {
    int major0;   // canonical start, major axis (ascending trace direction, [BRES]:19-29)
    int minor0;   // canonical start, minor axis
    int span;     // major-axis steps; the path has span+1 cells
    int inc;      // minor step direction ([BRES]:40-43)
    int hit_k;    // canonical index of the obstacle cell: span, or 0 when the trace was flipped
    int steep;    // major axis is y ([BRES]:14-17)
    double slope; // dy / float(dx) in float64 ([BRES]:35)
    int hx, hy;   // obstacle cell (the path's last element, [MAP]:44-45)
    int sx, sy;   // sensor cell (the path's first element)
};

enum BeamStatus { BEAM_OK = 0, BEAM_NOOP = 1, BEAM_NAN = 2, BEAM_TOO_LONG = 3, BEAM_INF_SKIP = 4, BEAM_OVERFLOW = 5 };

// [MAP]:33-36  int(S * (v + H)): float64 add, then multiply, then truncate toward zero.
__device__ __forceinline__ double cell_coord(double v, double cells_per_m, double off)
{
    return __dmul_rn(cells_per_m, __dadd_rn(v, off));
}

// Coordinates arrive as float64: float32 endpoints are upcast exactly by the callers, the fused
// ingestion path (ranges + pose) computes them in float64 like the reference does.
// The first half of the set-up: sensor and obstacle cells, the span and the beam's status (all that a bounding box
// needs; no division).
__device__ __forceinline__ int beam_cells(double fox, double foy, double fcx, double fcy, int xw, int yw,
                                          double cells_per_m, double off_x, double off_y, Beam &b)
{
    if (isinf(fox)) return BEAM_INF_SKIP;  // [MAP]:30 tests ox only
    if (isnan(fox) || isnan(foy) || isnan(fcx) || isnan(fcy)) return BEAM_NAN;  // int(nan): ValueError
    if (isinf(foy) || isinf(fcx) || isinf(fcy)) return BEAM_OVERFLOW;            // int(inf): OverflowError
    const double dxo = cell_coord(fox, cells_per_m, off_x), dyo = cell_coord(foy, cells_per_m, off_y);
    const double dxc = cell_coord(fcx, cells_per_m, off_x), dyc = cell_coord(fcy, cells_per_m, off_y);
    const double lim = 1073741824.0;  // 2^30: keeps every difference inside int32
    if (!(fabs(dxo) < lim && fabs(dyo) < lim && fabs(dxc) < lim && fabs(dyc) < lim)) return BEAM_TOO_LONG;
    const int x0 = __double2int_rz(dxc), y0 = __double2int_rz(dyc);  // sensor cell
    const int x1 = __double2int_rz(dxo), y1 = __double2int_rz(dyo);  // obstacle cell
    if (x0 == x1 && y0 == y1) return BEAM_NOOP;                      // [BRES]:10-11 empty path
    // no cell of the segment's bounding box inside the grid -> nothing to update
    if (max(x0, x1) < 0 || min(x0, x1) >= xw || max(y0, y1) < 0 || min(y0, y1) >= yw) return BEAM_NOOP;
    b.hx = x1;
    b.hy = y1;
    b.sx = x0;
    b.sy = y0;
    b.span = max(abs(x1 - x0), abs(y1 - y0));  // the major axis' extent
    if (b.span > B2S_MAX_PATH_CELLS) return BEAM_TOO_LONG;
    return BEAM_OK;
}

__device__ __forceinline__ int beam_setup(double fox, double foy, double fcx, double fcy, int xw, int yw,
                                          double cells_per_m, double off_x, double off_y, Beam &b)
{
    const int st = beam_cells(fox, foy, fcx, fcy, xw, yw, cells_per_m, off_x, off_y, b);
    if (st != BEAM_OK) return st;
    int x0 = b.sx, y0 = b.sy, x1 = b.hx, y1 = b.hy;
    const int steep = abs(y1 - y0) > abs(x1 - x0);
    if (steep) {
        int t = x0; x0 = y0; y0 = t;
        t = x1; x1 = y1; y1 = t;
    }
    const int flipped = x0 > x1;
    if (flipped) {
        int t = x0; x0 = x1; x1 = t;
        t = y0; y0 = y1; y1 = t;
    }
    b.major0 = x0;
    b.minor0 = y0;
    b.inc = (y0 < y1) ? 1 : -1;
    b.hit_k = flipped ? 0 : b.span;
    b.steep = steep;
    b.slope = __ddiv_rn((double)abs(y1 - y0), (double)b.span);
    return BEAM_OK;
}

__device__ __forceinline__ void count_status(int st, int32_t *counters)
{
    if (counters == nullptr) return;
    if (st == BEAM_NAN) atomicAdd(&counters[B2S_CNT_NONFINITE], 1);
    if (st == BEAM_OVERFLOW) atomicAdd(&counters[B2S_CNT_OVERFLOW], 1);
    if (st == BEAM_TOO_LONG) atomicAdd(&counters[B2S_CNT_TOO_LONG], 1);
    if (st == BEAM_INF_SKIP) atomicAdd(&counters[B2S_CNT_SKIPPED_INF], 1);
}

// One step of [BRES]:51-55.
__device__ __forceinline__ void bres_step(double &acc, int &minor, double slope, int inc)
{
    acc = __dadd_rn(acc, slope);
    if (acc >= 0.5) {
        minor += inc;
        acc = __dadd_rn(acc, -1.0);
    }
}

// ------------------------------------------------------------------------------------------
// Variant 1: one beam per thread, one RED.ADD per in-grid cell.

template <typename CT>
__global__ void __launch_bounds__(256)
grid_raycast_v1(int32_t *__restrict__ hit, int32_t *__restrict__ miss, int xw, int yw,
                double cells_per_m, double off_x, double off_y, const CT *__restrict__ ox,
                const CT *__restrict__ oy, const CT *__restrict__ cx,
                const CT *__restrict__ cy, long long total, int beams, int32_t *counters)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int s = (int)(i / beams);
    Beam b;
    const int st = beam_setup((double)__ldg(ox + i), (double)__ldg(oy + i), (double)__ldg(cx + s), (double)__ldg(cy + s), xw, yw,
                              cells_per_m, off_x, off_y, b);
    if (st != BEAM_OK) {
        count_status(st, counters);
        return;
    }
    const int wmaj = b.steep ? yw : xw, wmin = b.steep ? xw : yw;
    const int smaj = b.steep ? 1 : yw, smin = b.steep ? yw : 1;
    // in-grid window of the major axis; the recurrence is still replayed from k = 0
    const int k_lo = max(0, -b.major0);
    const int k_hi = min(b.span, wmaj - 1 - b.major0);
    double acc = 0.0;
    int minor = b.minor0;
    int k = 0;
    for (; k < k_lo; ++k) bres_step(acc, minor, b.slope, b.inc);
    for (; k <= k_hi; ++k) {
        if ((unsigned)minor < (unsigned)wmin) {
            const int cell = (b.major0 + k) * smaj + minor * smin;
            if (k == b.hit_k) atomicAdd(hit + cell, 1); else atomicAdd(miss + cell, 1);
        }
        bres_step(acc, minor, b.slope, b.inc);
    }
}

// ------------------------------------------------------------------------------------------
// Variant 2: warp-synchronous march with run aggregation.
//
// The 32 lanes of a warp hold 32 angularly adjacent beams of one scan.  All lanes advance one
// major-axis cell per iteration, lined up by distance from the sensor cell (a flipped trace
// starts at the obstacle, so it is delayed until it is `t` cells away from the sensor like its
// neighbours).  Adjacent beams share cells for the first ~1/(beam spacing) steps, and because
// they are sorted by angle, equal cells sit in adjacent lanes: one shuffle + ballot finds the
// runs and only the head lane of each run issues RED.ADD with the run length.

template <typename CT>
__global__ void __launch_bounds__(256)
grid_raycast_v2(int32_t *__restrict__ hit, int32_t *__restrict__ miss, int xw, int yw,
                double cells_per_m, double off_x, double off_y, const CT *__restrict__ ox,
                const CT *__restrict__ oy, const CT *__restrict__ cx,
                const CT *__restrict__ cy, long long total, int beams, int32_t *counters)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    Beam b;
    int st = BEAM_NOOP;
    if (i < total) {
        const int s = (int)(i / beams);
        st = beam_setup((double)__ldg(ox + i), (double)__ldg(oy + i), (double)__ldg(cx + s), (double)__ldg(cy + s), xw, yw,
                        cells_per_m, off_x, off_y, b);
        if (st != BEAM_OK) count_status(st, counters);
    }
    const bool live = (st == BEAM_OK);
    int span = live ? b.span : -1;
    int tmax = span;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tmax = max(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
    if (tmax < 0) return;

    const int wmaj = b.steep ? yw : xw, wmin = b.steep ? xw : yw;
    const int smaj = b.steep ? 1 : yw, smin = b.steep ? yw : 1;
    // canonical index k = t - delay; a flipped trace ends at the sensor cell when t == tmax
    const int delay = (live && b.hit_k == 0) ? (tmax - span) : 0;
    double acc = 0.0;
    int minor = live ? b.minor0 : 0;
    const int dead_key = -1 - lane;  // unique per lane: never equal to a neighbour's cell

    for (int t = 0; t <= tmax; ++t) {
        const int k = t - delay;
        const bool on = live && k >= 0 && k <= span;
        int key = dead_key;
        if (on) {
            const int major = b.major0 + k;
            if ((unsigned)major < (unsigned)wmaj && (unsigned)minor < (unsigned)wmin) {
                const int cell = major * smaj + minor * smin;
                if (k == b.hit_k) atomicAdd(hit + cell, 1);  // once per beam
                else key = cell;
            }
            bres_step(acc, minor, b.slope, b.inc);
        }
        const int left = __shfl_up_sync(0xffffffffu, key, 1);
        const bool head = (lane == 0) || (key != left);
        const unsigned heads = __ballot_sync(0xffffffffu, head);
        if (head && key >= 0) {
            const unsigned rest = (lane == 31) ? 0u : (heads >> (lane + 1));
            const int run = rest ? __ffs(rest) : (32 - lane);
            atomicAdd(miss + key, run);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Variant 3: the march of variant 2 with a lean inner loop (the kernel is issue-bound: ncu shows
// 77% issue-slot utilisation and <10% FP64 pipe for v2, so every instruction per step counts).
//   * the endpoint hit is one RED per beam taken straight from the obstacle cell, outside the loop
//   * per-lane emission window [t_em, t_em + em_len] in warp time replaces the per-step bounds tests
//     on the major axis; the minor axis is tested on the pre-multiplied cell offset
//   * cell offsets advance incrementally (no multiplies in the loop)
//   * flipped traces need a "not started yet" guard only while some lane is still waiting
//     (phase A); once every lane has started the guard disappears (phase B)
//   * run length = clz of the reversed head mask, RED predicated instead of branched

template <bool GUARD_START>
__device__ __forceinline__ void march_step(int t, int delay, double slope, double &acc, unsigned &cmaj, int &minor,
                                           unsigned smaj, int smin, int inc, unsigned wmin, int t_em,
                                           unsigned em_len, int dead_key, unsigned lane, unsigned lane_bit,
                                           int32_t *__restrict__ miss)
{
    const bool started = !GUARD_START || (t >= delay);
    const bool emit = ((unsigned)(t - t_em) <= em_len) && ((unsigned)minor < wmin);
    // inside the window the true offset is in [0, xw*yw): modular arithmetic on cmaj is exact there
    const int key = emit ? (int)(cmaj + (unsigned)(minor * smin)) : dead_key;
    if (started) {
        acc = __dadd_rn(acc, slope);  // [BRES]:51
        if (acc >= 0.5) {             // [BRES]:53
            minor += inc;             // [BRES]:54
            acc = __dadd_rn(acc, -1.0);  // [BRES]:55
        }
        cmaj += smaj;
    }
    const int left = __shfl_up_sync(0xffffffffu, key, 1);
    const bool head = (lane == 0) || (key != left);
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    // lanes after this one up to the next head carry the same cell: run = distance to that head
    const unsigned ahead = ((__brev(heads) << lane) << 1) | lane_bit;
    const int run = __clz(ahead) + 1;
    if (head && emit) atomicAdd(miss + key, run);
}

template <typename CT>
__global__ void __launch_bounds__(256)
grid_raycast_v3(int32_t *__restrict__ hit, int32_t *__restrict__ miss, int xw, int yw,
                double cells_per_m, double off_x, double off_y, const CT *__restrict__ ox,
                const CT *__restrict__ oy, const CT *__restrict__ cx,
                const CT *__restrict__ cy, long long total, int beams, int32_t *counters)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned lane = threadIdx.x & 31;
    Beam b;
    b.major0 = b.minor0 = b.span = b.inc = b.hit_k = b.steep = b.hx = b.hy = b.sx = b.sy = 0;
    b.slope = 0.0;
    int st = BEAM_NOOP;
    if (i < total) {
        const int s = (int)(i / beams);
        st = beam_setup((double)__ldg(ox + i), (double)__ldg(oy + i), (double)__ldg(cx + s), (double)__ldg(cy + s), xw, yw,
                        cells_per_m, off_x, off_y, b);
        if (st != BEAM_OK) count_status(st, counters);
    }
    const bool live = (st == BEAM_OK);
    const int span = live ? b.span : -1;
    int tmax = span;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tmax = max(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
    if (tmax < 0) return;

    // endpoint: the obstacle cell is the last path element whenever the path is not empty
    if (live && (unsigned)b.hx < (unsigned)xw && (unsigned)b.hy < (unsigned)yw)
        atomicAdd(hit + (b.hx * yw + b.hy), 1);

    const int wmaj = b.steep ? yw : xw;
    const unsigned wmin = (unsigned)(b.steep ? xw : yw);
    const unsigned smaj = b.steep ? 1u : (unsigned)yw;
    const int smin = b.steep ? yw : 1;
    // canonical index k = t - delay; a flipped trace reaches the sensor cell at t == tmax
    const int delay = (live && b.hit_k == 0) ? (tmax - span) : 0;
    int dmax = delay;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dmax = max(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    // emission window in canonical k: inside the grid on the major axis, obstacle cell excluded
    int k_lo = max(0, -b.major0), k_hi = min(span, wmaj - 1 - b.major0);
    if (b.hit_k == 0) k_lo = max(k_lo, 1); else k_hi = min(k_hi, span - 1);
    const bool any = live && k_hi >= k_lo;
    const int t_em = any ? delay + k_lo : 0x3fffffff;
    const unsigned em_len = any ? (unsigned)(k_hi - k_lo) : 0u;

    double acc = 0.0;
    unsigned cmaj = (unsigned)b.major0 * smaj;  // major part of the cell offset at k = 0 (mod 2^32)
    int minor = b.minor0;
    const int inc = b.inc;
    const int dead_key = -1 - (int)lane;  // unique per lane: never equal to a neighbour's cell
    const unsigned lane_bit = 1u << lane;
    const double slope = b.slope;

    int t = 0;
    for (; t < dmax; ++t)
        march_step<true>(t, delay, slope, acc, cmaj, minor, smaj, smin, inc, wmin, t_em, em_len, dead_key, lane,
                         lane_bit, miss);
#pragma unroll 4
    for (; t <= tmax; ++t)
        march_step<false>(t, delay, slope, acc, cmaj, minor, smaj, smin, inc, wmin, t_em, em_len, dead_key, lane,
                          lane_bit, miss);
}

// ------------------------------------------------------------------------------------------
// Variant 4: variant 3 plus a transposed scratch plane for the steep (y-major) beams.
//
// Measured on B200 (profiles/microbench): RED.ADD costs ~1.5 SM-cycles per distinct 32-byte sector a
// warp instruction touches, not per lane -- 32 lanes on consecutive words retire in ~7 cycles, 32
// scattered lanes in ~50.  In the [x][y] planes the run heads of a warp of x-major beams sit on
// consecutive y (a few sectors per step), but those of y-major beams are a whole row apart (one
// sector each), and they dominate the RED time of variants 2/3.  Here y-major beams accumulate
// into a scratch plane stored [y][x], where THEIR heads are consecutive too; a tiled transpose-add
// then folds the touched bounding box of the scratch plane into `miss` and re-zeroes it.
// Integer adds commute, so the result is bit-identical.

struct GridWorkspace {      // lives at the front of the caller-provided workspace (GRID_WS_HEADER bytes)
    int bbox[4];            // atomicMax of (-xmin, xmax, -ymin, ymax) over warps with y-major beams; reset to very negative
    int pad[12];
};
static_assert(sizeof(GridWorkspace) == GRID_WS_HEADER, "workspace header size");
// layout of the workspace: [GridWorkspace][dirty map: 1 byte per 64x64 tile, padded to 256 B][scratch plane [yw][xw]]

// One warp-step.  Everything that addresses memory is kept DOUBLED (key2 = 2*cell + plane bit) so the
// run key, the plane selector and the byte offset (key2 * 2, minus the plane bit folded into the
// base pointer) come out of one add; SHFL's own in-range predicate marks lane 0 as a run head;
// the run length is ffs of the head mask funnel-shifted past this lane with a sentinel at lane 32;
// the RED is predicated, not branched.
//
// CORE = true is the same step for the part of the march where NOTHING has to be tested: every lane of the warp is
// live, started, inside its emission window and inside the grid (see grid_raycast_v4), so the window compare, the
// clip test and the dead-key select disappear -- 6 of the 34 issue slots of a step.
template <bool GUARD_START, int SIGN, bool CORE = false>
__device__ __forceinline__ void march_step4(int t, int delay, double slope, double &acc, unsigned &cmaj2, int &minor2,
                                            unsigned pitch2, int inc2, unsigned wmin2, int t_em, unsigned em_len,
                                            unsigned dead_key, unsigned lane1, unsigned long long plane_base)
{
    const bool emit = CORE || (((unsigned)(t - t_em) <= em_len) && ((unsigned)minor2 < wmin2));
    const unsigned key = emit ? (cmaj2 + (unsigned)minor2) : dead_key;  // exact inside the window
    if (!GUARD_START || t >= delay) {
        // [BRES]:51-55, kept as predicated instructions (the compiler otherwise turns the `if` into
        // an unconditional DADD plus selects): acc += slope; if (acc >= 0.5) { minor += inc; acc -= 1.0; }
        asm("{\n\t"
            ".reg .pred p;\n\t"
            "add.rn.f64 %0, %0, %2;\n\t"
            "setp.ge.f64 p, %0, 0d3FE0000000000000;\n\t"
            "@p add.rn.f64 %0, %0, 0dBFF0000000000000;\n\t"
            "@p add.s32 %1, %1, %3;\n\t"
            "}"
            : "+d"(acc), "+r"(minor2)
            : "d"(slope), "r"(inc2));
        cmaj2 += pitch2;
    }
    unsigned left;
    int in_range;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "shfl.sync.up.b32 %0|p, %2, 1, 0, 0xffffffff;\n\t"
        "selp.s32 %1, 1, 0, p;\n\t"
        "}"
        : "=r"(left), "=r"(in_range)
        : "r"(key));
    const bool head = !in_range || (key != left);
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    // heads of the lanes after this one, with a sentinel head at virtual lane 32
    const int run = SIGN * __ffs(__funnelshift_rc(heads, 1u, lane1));
    // byte offset of the int32 cell = (key >> 1) * 4 = key * 2 - 2 * (plane bit); the latter is folded into plane_base
    const unsigned long long addr = plane_base + (unsigned long long)key * 2ull;
    asm volatile(
        "{\n\t"
        ".reg .pred q;\n\t"
        "setp.ne.s32 q, %2, 0;\n\t"
        "@q red.global.add.s32 [%0], %1;\n\t"
        "}" ::"l"(addr),
        "r"(run), "r"((int)(head && emit))
        : "memory");
}

// Where a beam's endpoints come from.  IN_F32 / IN_F64: world-frame endpoints ox, oy + sensor position
// cx, cy (the arguments of Mapping.update) as float32, or as the float64 the reference's callers pass
// ([SLAM]:89-90: obs and xEst are float64).  IN_FUSED: raw ranges + pose, i.e. the node's
// laserToNumpy ([SLAM]:115-123) and `u2T(xEst).dot(np_msg)` ([SLAM]:130-137,89) evaluated per beam in
// float64: p = (cos a * r, sin a * r) with inf -> clamp, o = (cw*px + (-sw)*py) + x, (sw*px + cw*py) + y.
// cos/sin of the beam angles and of the yaw are computed by the host exactly as the reference
// computes them (NumPy / math), so the device only multiplies and adds.
enum { IN_F32 = 0, IN_FUSED = 1, IN_F64 = 2 };
struct ScanInput {
    const void *ox, *oy, *cx, *cy;   // endpoints modes: float32 (IN_F32) or float64 (IN_F64, the reference's dtype)
    const float *ranges;             // fused mode: [scans][beams]
    const double *pose4;             // fused mode: [scans][4] = x, y, cos(yaw), sin(yaw)
    const double *beam_cs;           // fused mode: [beams][2] = cos(angle), sin(angle)
    double clamp;                    // fused mode: replacement for +inf ranges (MAX_LASER_RANGE), <= 0: none
};

template <int MODE>
__device__ __forceinline__ void load_beam(const ScanInput &in, long long i, int beams, double &fox, double &foy,
                                          double &fcx, double &fcy)
{
    // (a 64-bit division costs ~70 instructions; every launch of a realistic size fits 32 bits)
    const int s = (i >> 32) == 0 ? (int)((unsigned)i / (unsigned)beams) : (int)(i / beams);
    if (MODE == IN_F32) {
        fox = (double)__ldg((const float *)in.ox + i);
        foy = (double)__ldg((const float *)in.oy + i);
        fcx = (double)__ldg((const float *)in.cx + s);
        fcy = (double)__ldg((const float *)in.cy + s);
    } else if (MODE == IN_F64) {  // [MAP]:33-36 consumes float64: nothing is narrowed on the way to int()
        fox = __ldg((const double *)in.ox + i);
        foy = __ldg((const double *)in.oy + i);
        fcx = __ldg((const double *)in.cx + s);
        fcy = __ldg((const double *)in.cy + s);
    } else {
        const int j = (int)(i - (long long)s * beams);
        double r = (double)__ldg(in.ranges + i);
        if (in.clamp > 0.0 && r == INFINITY) r = in.clamp;  // [SLAM]:119 (only +inf compares equal)
        const double2 cs = __ldg(reinterpret_cast<const double2 *>(in.beam_cs) + j);
        const double px = __dmul_rn(cs.x, r), py = __dmul_rn(cs.y, r);  // [SLAM]:122
        const double2 xy = __ldg(reinterpret_cast<const double2 *>(in.pose4) + 2 * s);
        const double2 cw = __ldg(reinterpret_cast<const double2 *>(in.pose4) + 2 * s + 1);
        fox = __dadd_rn(__dadd_rn(__dmul_rn(cw.x, px), __dmul_rn(-cw.y, py)), xy.x);  // [SLAM]:134,89
        foy = __dadd_rn(__dadd_rn(__dmul_rn(cw.y, px), __dmul_rn(cw.x, py)), xy.y);   // [SLAM]:135,89
        fcx = xy.x;
        fcy = xy.y;
    }
}

// The march of variants 4 / 5 for one warp: lane l ray-casts beam i (flat index scan * beams + beam) when `valid`.
// All 32 lanes call it together.  SIGN = +1 applies a batch, SIGN = -1 takes the same batch back out (exact inverse:
// integer adds).
template <int SIGN, int MODE, bool CORE_PHASE>
__device__ __forceinline__ void raycast_warp_v4(int32_t *__restrict__ hit, int32_t *__restrict__ miss,
                                                int32_t *__restrict__ scratch_t, GridWorkspace *__restrict__ ws,
                                                uint8_t *__restrict__ dirty, int xw, int yw, double cells_per_m,
                                                double off_x, double off_y, const ScanInput &in, long long i, bool valid,
                                                int beams, int32_t *counters)
{
    const unsigned lane = threadIdx.x & 31;
    Beam b;
    b.major0 = b.minor0 = b.span = b.inc = b.hit_k = b.steep = b.hx = b.hy = b.sx = b.sy = 0;
    b.slope = 0.0;
    int st = BEAM_NOOP;
    if (valid) {
        double fox, foy, fcx, fcy;
        load_beam<MODE>(in, i, beams, fox, foy, fcx, fcy);
        st = beam_setup(fox, foy, fcx, fcy, xw, yw, cells_per_m, off_x, off_y, b);
        if (st != BEAM_OK && SIGN > 0) count_status(st, counters);
    }
    const bool live = (st == BEAM_OK);
    const int span = live ? b.span : -1;
    // (warp reductions are single REDUX instructions: the set-up of a warp used to spend 45 shuffles on them)
    const int tmax = __reduce_max_sync(0xffffffffu, span);
    if (tmax < 0) return;

    if (live && (unsigned)b.hx < (unsigned)xw && (unsigned)b.hy < (unsigned)yw)
        atomicAdd(hit + (b.hx * yw + b.hy), SIGN);

    // Bounding box (clipped to the grid) of everything this warp can touch.  It marks the 64 x 64-cell
    // tiles the warp dirties (sparse zeroing / merging of the planes downstream) and, when the warp
    // holds y-major beams, bounds the part of the transposed scratch plane that has to be folded back.
    {
        const int very_neg = (int)0x80808080;
        int nx0 = very_neg, x1 = very_neg, ny0 = very_neg, y1 = very_neg;
        if (live) {
            nx0 = -max(0, min(b.sx, b.hx));
            x1 = min(xw - 1, max(b.sx, b.hx));
            ny0 = -max(0, min(b.sy, b.hy));
            y1 = min(yw - 1, max(b.sy, b.hy));
        }
        nx0 = __reduce_max_sync(0xffffffffu, nx0);
        x1 = __reduce_max_sync(0xffffffffu, x1);
        ny0 = __reduce_max_sync(0xffffffffu, ny0);
        y1 = __reduce_max_sync(0xffffffffu, y1);
        if (__any_sync(0xffffffffu, live && b.steep) && lane < 4) {
            // lane k widens bound k, and only when it actually does: after the first few warps of a launch almost
            // none does, and half a million warps no longer queue up on the same four words (a stale read only
            // costs a redundant atomic)
            const int mine = lane == 0 ? nx0 : lane == 1 ? x1 : lane == 2 ? ny0 : y1;
            if (mine > *reinterpret_cast<volatile int *>(&ws->bbox[lane])) atomicMax(&ws->bbox[lane], mine);
        }
        const int tx0 = (-nx0) / GRID_TILE, tx1 = x1 / GRID_TILE, ty0 = (-ny0) / GRID_TILE, ty1 = y1 / GRID_TILE;
        const int ny = ty1 - ty0 + 1, cnt = (tx1 - tx0 + 1) * ny, tiles_y = grid_tiles(yw);
        for (int k = lane; k < cnt; k += 32) dirty[(tx0 + k / ny) * tiles_y + ty0 + k % ny] = 1;
    }

    const int wmaj = b.steep ? yw : xw;
    const unsigned wmin = (unsigned)(b.steep ? xw : yw);
    const unsigned steep_bit = b.steep ? 1u : 0u;
    // both planes are stored major-row by major-row for their beams; offsets are kept doubled
    const unsigned pitch2 = 2u * wmin;
    const unsigned long long plane_base = (unsigned long long)(uintptr_t)(b.steep ? scratch_t : miss) - 2ull * steep_bit;
    const int delay = (live && b.hit_k == 0) ? (tmax - span) : 0;
    const int dmax = __reduce_max_sync(0xffffffffu, delay);
    int k_lo = max(0, -b.major0), k_hi = min(span, wmaj - 1 - b.major0);
    if (b.hit_k == 0) k_lo = max(k_lo, 1); else k_hi = min(k_hi, span - 1);
    const bool any = live && k_hi >= k_lo;
    const int t_em = any ? delay + k_lo : 0x3fffffff;
    const unsigned em_len = any ? (unsigned)(k_hi - k_lo) : 0u;

    double acc = 0.0;
    unsigned cmaj2 = (unsigned)b.major0 * pitch2 + steep_bit;  // 2 * (major part of the cell offset) + plane bit
    // |minor0| < 2^30, so 2 * minor0 fits an int; only values in [0, 2 * wmin) ever reach memory
    int minor2 = 2 * b.minor0;
    const int inc2 = 2 * b.inc;
    const unsigned wmin2 = 2u * wmin;
    const unsigned dead_key = 0x80000000u | lane;  // cells < 2^30, so live keys stay below 2^31
    const unsigned lane1 = lane + 1;
    const double slope = b.slope;

    // Core phase (variant 5): warp times [c_lo, c_hi] in which every lane emits -- after the last lane has started and
    // entered its window, before the first lane leaves its window -- provided all 32 lanes are live and none of their
    // rays is clipped by the grid.  Typically 80-85 % of a warp's steps (beams of a warp differ in length by ~15 %).
    int c_lo = 0x3fffffff, c_hi = -1;
    if (CORE_PHASE) {
        const bool unclipped = live && min(b.sx, b.hx) >= 0 && max(b.sx, b.hx) < xw && min(b.sy, b.hy) >= 0 &&
                               max(b.sy, b.hy) < yw;
        const int lo = __reduce_max_sync(0xffffffffu, any ? t_em : 0x3fffffff);
        const int hi = __reduce_min_sync(0xffffffffu, any ? t_em + (int)em_len : -1);
        if (__all_sync(0xffffffffu, unclipped && any)) {
            c_lo = max(lo, dmax);
            c_hi = hi;
        }
    }

    int t = 0;
    for (; t < dmax; ++t)
        march_step4<true, SIGN>(t, delay, slope, acc, cmaj2, minor2, pitch2, inc2, wmin2, t_em, em_len, dead_key, lane1,
                          plane_base);
    if (CORE_PHASE && c_lo <= c_hi) {
        for (; t < c_lo; ++t)
            march_step4<false, SIGN>(t, delay, slope, acc, cmaj2, minor2, pitch2, inc2, wmin2, t_em, em_len, dead_key,
                                     lane1, plane_base);
#pragma unroll 4
        for (; t <= c_hi; ++t)
            march_step4<false, SIGN, true>(t, delay, slope, acc, cmaj2, minor2, pitch2, inc2, wmin2, t_em, em_len,
                                           dead_key, lane1, plane_base);
    }
#pragma unroll 4
    for (; t <= tmax; ++t)
        march_step4<false, SIGN>(t, delay, slope, acc, cmaj2, minor2, pitch2, inc2, wmin2, t_em, em_len, dead_key, lane1,
                           plane_base);
}

template <int SIGN, int MODE, bool CORE_PHASE>
__global__ void __launch_bounds__(256, 8)
grid_raycast_v4(int32_t *__restrict__ hit, int32_t *__restrict__ miss, int32_t *__restrict__ scratch_t,
                GridWorkspace *__restrict__ ws, uint8_t *__restrict__ dirty, int xw, int yw, double cells_per_m,
                double off_x, double off_y, const ScanInput in, long long total, int beams, int32_t *counters)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    raycast_warp_v4<SIGN, MODE, CORE_PHASE>(hit, miss, scratch_t, ws, dirty, xw, yw, cells_per_m, off_x, off_y, in, i,
                                            i < total, beams, counters);
}

// ------------------------------------------------------------------------------------------
// Variant 6 (default): consecutive scans counted in a shared-memory tile.
//
// The scans of a trajectory overlap: consecutive scans are a few cells apart and each covers a disk of 60-200 cells,
// so V6_SCANS consecutive scans visit almost the same cells.  A CTA takes V6_SCANS consecutive scans x one sector of
// V6_SECTOR adjacent beams, finds the bounding box of everything they touch, and -- when that box fits the tile and
// no ray is clipped by the grid -- counts every visit with an unpredicated shared atomicAdd (ATOMS.POPC.INC: lanes on
// the same word merge in hardware, no run finding, no divergent region), then adds the tile to `miss` with coalesced
// full-warp REDs.  Each lane marches its own beam with the reference's float64 recurrence; lanes need not move in
// step.  A CTA whose box does not fit, or that has a clipped ray, runs the variant-5 march for its beams instead
// (random scans, map edges), so any input stays exact.  Integer adds commute: the counts are those of variant 5.
//
// A CTA's beams form 32 warp-units: 32 adjacent beams of one scan each (unit u: scan u / 2, beams 32 * (u & 1) ..
// + 31 of the sector).  Layout 1 (default) runs 512 threads, two units per warp: the box pass measures each unit's
// longest beam, and warp w marches the unit of rank w, then that of rank 31 - w (longest with shortest).  The scans of
// a CTA differ in length by up to 2x, and the CTA holds its tile until its last warp is done; pairing brings the
// warps' march lengths within a few percent of each other.  Layout 0 runs 1024 threads, one unit per warp, in order.
constexpr int V6_SCANS = 16;
constexpr int V6_SECTOR = 64;     // beams; two units of one scan
constexpr int V6_UNITS = V6_SCANS * V6_SECTOR / 32;
constexpr int V6_TILE_WORDS = 27 * 1024;  // 108 KB: two CTAs per SM
int g_grid_tile_layout = 1;

#ifdef B2S_GRID_PHASES
// Diagnostic build only (profiles/scripts/grid_phases.py): per CTA, V6_PHASE_WORDS clock64 stamps.  Word 0: %smid,
// 1..5: start, box known, tile zeroed, march done, end; 6: 1 when the CTA fell back; 7: warps; 8 + w: warp w's march end.
constexpr int V6_PHASE_WORDS = 8 + V6_UNITS;
__device__ unsigned long long *g_grid_phases;
extern "C" int b2s_grid_phases_buffer(void *rec)
{
    B2S_CUDA(cudaMemcpyToSymbol(g_grid_phases, &rec, sizeof(rec)));
    return B2S_OK;
}
#define V6_STAMP(word, value)                                                                                      \
    do {                                                                                                           \
        if (g_grid_phases) g_grid_phases[(size_t)blockIdx.x * V6_PHASE_WORDS + (word)] = (value);                 \
    } while (0)
#else
#define V6_STAMP(word, value) do { } while (0)
#endif

// [BRES]:51-55 on a shared-memory byte address: acc += slope; if (acc >= 0.5) { addr += dmin; acc -= 1.0; } addr += dmaj.
// For a finite acc, acc >= 0.5 exactly when the high word, read as a signed int, is >= 0x3FE00000 (0.5 has a zero low
// word; negative values and -0.0 have the sign bit set).  acc - 0.0 == acc bit for bit (-0.0 included), so subtracting
// c = 1.0 or 0.0, built from one select on its high word, is the reference's conditional acc -= 1.0: one integer
// compare instead of an FP64 one, and the second DADD needs no select after it.
__device__ __forceinline__ void tile_step(double &acc, unsigned &addr, double slope, unsigned dmin, unsigned dmaj)
{
    acc = __dadd_rn(acc, slope);
    const bool up = __double2hiint(acc) >= 0x3FE00000;
    acc = __dsub_rn(acc, __hiloint2double(up ? 0x3FF00000 : 0, 0));
    if (up) addr += dmin;
    addr += dmaj;
}

// One beam's misses into the tile: word (x - bx) * pitch + (y - by) counts cell (x, y); the box holds the whole path.
__device__ __forceinline__ void march_tile(const Beam &b, unsigned tile_base, int bx, int by, int pitch)
{
    // tile word of the canonical start; the major axis advances by dmaj bytes per step, the minor axis by dmin
    const int mx = b.steep ? b.minor0 : b.major0, my = b.steep ? b.major0 : b.minor0;
    unsigned addr = tile_base + 4u * (unsigned)((mx - bx) * pitch + (my - by));
    const unsigned dmaj = 4u * (b.steep ? 1u : (unsigned)pitch);
    const unsigned dmin = 4u * (unsigned)(b.steep ? b.inc * pitch : b.inc);
    const double slope = b.slope;
    double acc = 0.0;
    // the path is k = 0 .. span; every cell but the obstacle's (k = hit_k: span, or 0 when flipped) is a miss
    if (b.hit_k == 0) tile_step(acc, addr, slope, dmin, dmaj);
    // unpredicated: ATOMS.POPC.INC, lanes on one word merge (a predicated shared atomic becomes a divergent region)
#pragma unroll 4
    for (int n = b.span; n > 0; --n) {
        asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(addr) : "memory");
        tile_step(acc, addr, slope, dmin, dmaj);
    }
}

// Flat index of this lane's beam in unit u of the CTA whose first scan is s0 and first beam b0; false past the input.
__device__ __forceinline__ bool v6_beam(int u, int s0, int b0, int scans, int beams, long long &i)
{
    const int s = s0 + (u >> 1), bm = b0 + 32 * (u & 1) + (int)(threadIdx.x & 31);
    i = (long long)s * beams + bm;
    return s < scans && bm < beams;
}

// UNITS: warp-units per warp (layout 0: 1, layout 1: 2).
template <int MODE, int UNITS>
__global__ void __launch_bounds__(V6_UNITS * 32 / UNITS, 2)
grid_raycast_v6(int32_t *__restrict__ hit, int32_t *__restrict__ miss, int32_t *__restrict__ scratch_t,
                GridWorkspace *__restrict__ ws, uint8_t *__restrict__ dirty, int xw, int yw, double cells_per_m,
                double off_x, double off_y, const ScanInput in, int scans, int beams, int32_t *counters)
{
    static_assert(UNITS == 1 || UNITS == 2, "a warp marches one unit, or a long and a short one");
    constexpr int NWARPS = V6_UNITS / UNITS;
    extern __shared__ uint32_t tile[];
    __shared__ int box[5];  // -xmin, xmax, -ymin, ymax over the live beams (max-reduced), clipped flag
    __shared__ int unit_span[V6_UNITS];  // longest live beam of each unit, -1 if none (layout 1)
    __shared__ int order[V6_UNITS];      // units by decreasing span, ties by index (layout 1)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#ifdef B2S_GRID_PHASES
    if (threadIdx.x == 0) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        V6_STAMP(0, smid);
        V6_STAMP(1, clock64());
        V6_STAMP(7, NWARPS);
    }
#endif
    const int sectors = (beams + V6_SECTOR - 1) / V6_SECTOR;
    const int s0 = (int)(blockIdx.x / sectors) * V6_SCANS, b0 = (int)(blockIdx.x % sectors) * V6_SECTOR;
    if (threadIdx.x < 5) box[threadIdx.x] = threadIdx.x < 4 ? (int)0x80808080 : 0;
    __syncthreads();

    // ---- box pass: bounding box of the sensor and obstacle cells of the live beams, whether any ray is clipped, and
    // each unit's longest beam.  Cells only: the division of the set-up is left to the march.
    {
        const int very_neg = (int)0x80808080;
        int nx0 = very_neg, x1 = very_neg, ny0 = very_neg, y1 = very_neg;
        bool clipped = false;
#pragma unroll
        for (int k = 0; k < UNITS; ++k) {
            const int u = warp + k * NWARPS;
            long long i;
            int span = -1;
            if (v6_beam(u, s0, b0, scans, beams, i)) {
                double fox, foy, fcx, fcy;
                load_beam<MODE>(in, i, beams, fox, foy, fcx, fcy);
                Beam b;
                if (beam_cells(fox, foy, fcx, fcy, xw, yw, cells_per_m, off_x, off_y, b) == BEAM_OK) {
                    nx0 = max(nx0, -min(b.sx, b.hx));
                    x1 = max(x1, max(b.sx, b.hx));
                    ny0 = max(ny0, -min(b.sy, b.hy));
                    y1 = max(y1, max(b.sy, b.hy));
                    clipped |= min(b.sx, b.hx) < 0 || max(b.sx, b.hx) >= xw || min(b.sy, b.hy) < 0 ||
                               max(b.sy, b.hy) >= yw;
                    span = b.span;
                }
            }
            if (UNITS > 1) {
                span = __reduce_max_sync(0xffffffffu, span);
                if (lane == 0) unit_span[u] = span;
            }
        }
        nx0 = __reduce_max_sync(0xffffffffu, nx0);
        x1 = __reduce_max_sync(0xffffffffu, x1);
        ny0 = __reduce_max_sync(0xffffffffu, ny0);
        y1 = __reduce_max_sync(0xffffffffu, y1);
        clipped = __any_sync(0xffffffffu, clipped);
        if (lane < 4) atomicMax(&box[lane], lane == 0 ? nx0 : lane == 1 ? x1 : lane == 2 ? ny0 : y1);
        if (lane == 4 && clipped) box[4] = 1;
    }
    __syncthreads();
    const int bx = -box[0], by = -box[2];
    const bool empty = box[1] < 0;  // no live beam: nothing but status counts
    const int w = empty ? 0 : box[1] - bx + 1, h = empty ? 0 : box[3] - by + 1;
    const int pitch = h | 1;  // odd: the words of a y-major warp (one per row) spread over all banks
    if (threadIdx.x == 0) V6_STAMP(2, clock64());
    if (box[4] || (long long)w * pitch > V6_TILE_WORDS) {
        if (threadIdx.x == 0) V6_STAMP(6, 1);
#pragma unroll 1
        for (int k = 0; k < UNITS; ++k) {
            long long i;
            const bool valid = v6_beam(warp + k * NWARPS, s0, b0, scans, beams, i);
            raycast_warp_v4<1, MODE, true>(hit, miss, scratch_t, ws, dirty, xw, yw, cells_per_m, off_x, off_y, in, i,
                                           valid, beams, counters);
        }
#ifdef B2S_GRID_PHASES
        __syncthreads();
        if (threadIdx.x == 0) V6_STAMP(5, clock64());
#endif
        return;
    }

    // ---- private path: the box lies inside the grid
    if (UNITS > 1 && warp == 0) {
        const int mine = unit_span[lane];
        int rank = 0;
        for (int u = 0; u < V6_UNITS; ++u) {
            const int o = unit_span[u];
            rank += (o > mine) || (o == mine && u < lane);
        }
        order[rank] = lane;
    }
    for (int k = threadIdx.x; k < w * pitch; k += NWARPS * 32) tile[k] = 0;
    if (!empty) {
        const int tx0 = bx / GRID_TILE, ty0 = by / GRID_TILE, ny = box[3] / GRID_TILE - ty0 + 1;
        const int cnt = ((bx + w - 1) / GRID_TILE - tx0 + 1) * ny, tiles_y = grid_tiles(yw);
        for (int k = threadIdx.x; k < cnt; k += NWARPS * 32) dirty[(tx0 + k / ny) * tiles_y + ty0 + k % ny] = 1;
    }
    __syncthreads();
    if (threadIdx.x == 0) V6_STAMP(3, clock64());
#pragma unroll 1
    for (int k = 0; k < UNITS; ++k) {
        const int u = UNITS == 1 ? warp : order[k == 0 ? warp : V6_UNITS - 1 - warp];
        long long i;
        if (v6_beam(u, s0, b0, scans, beams, i)) {
            double fox, foy, fcx, fcy;
            load_beam<MODE>(in, i, beams, fox, foy, fcx, fcy);
            Beam b;
            const int st = beam_setup(fox, foy, fcx, fcy, xw, yw, cells_per_m, off_x, off_y, b);
            if (st == BEAM_OK) {
                atomicAdd(hit + (b.hx * yw + b.hy), 1);  // the obstacle cell: last path element, inside the grid here
                march_tile(b, smem_addr(tile), bx, by, pitch);
            } else {
                count_status(st, counters);
            }
        }
    }
#ifdef B2S_GRID_PHASES
    __syncwarp();
    if (lane == 0) V6_STAMP(8 + warp, clock64());
#endif
    __syncthreads();
    if (threadIdx.x == 0) V6_STAMP(4, clock64());

    // ---- flush: each warp takes whole rows of the box and adds them in 32-cell segments aligned in the plane, loading
    // four segments before it issues their REDs; all-zero segments are skipped
    const int g0 = by >> 5, nseg = empty ? 0 : ((by + h - 1) >> 5) - g0 + 1;
    for (int r = warp; r < w; r += NWARPS) {
        const uint32_t *row = tile + r * pitch;
        int32_t *mrow = miss + (size_t)(bx + r) * yw;
        for (int g = 0; g < nseg; g += 4) {
            int v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int y = ((g0 + g + j) << 5) + lane;
                v[j] = (g + j < nseg && y >= by && y < by + h) ? (int)row[y - by] : 0;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (__any_sync(0xffffffffu, v[j] != 0)) {
                    // every lane adds (0 outside the box); past the last column it adds to a cell of its own row
                    const int y = ((g0 + g + j) << 5) + lane;
                    asm volatile("red.global.add.s32 [%0], %1;" ::"l"(mrow + min(y, yw - 1)), "r"(v[j]) : "memory");
                }
            }
        }
    }
#ifdef B2S_GRID_PHASES
    __syncthreads();
    if (threadIdx.x == 0) V6_STAMP(5, clock64());
#endif
}

// miss[x][y] += scratch_t[y][x] over the recorded bounding box, scratch_t cleared on the way.
// A fixed-size grid walks the 32 x 32-cell tiles INSIDE the box (a 16384^2 plane has 262 144 such tiles, a step
// touches a few thousand of them: launching one CTA per tile of the plane cost more than the fold itself).
__global__ void __launch_bounds__(256)
grid_fold_kernel(int32_t *__restrict__ miss, int32_t *__restrict__ scratch_t, const GridWorkspace *__restrict__ ws,
                 int xw, int yw)
{
    __shared__ int tile[32][33];
    const int xmin = -ws->bbox[0], xmax = ws->bbox[1], ymin = -ws->bbox[2], ymax = ws->bbox[3];
    if (xmax < 0 || ymax < 0) return;  // no y-major beam in this launch
    const int bx0 = xmin >> 5, by0 = ymin >> 5;
    const int nbx = (xmax >> 5) - bx0 + 1, nby = (ymax >> 5) - by0 + 1;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    for (int t = blockIdx.x; t < nbx * nby; t += gridDim.x) {
        const int x0 = (bx0 + t / nby) * 32, y0 = (by0 + t % nby) * 32;
        int any_nz = 0;
#pragma unroll
        for (int r = ty; r < 32; r += 8) {
            const int y = y0 + r, x = x0 + tx;
            int v = 0;
            if (y < yw && x < xw) {
                const size_t at = (size_t)y * xw + x;
                v = scratch_t[at];
                if (v) scratch_t[at] = 0;
            }
            tile[r][tx] = v;
            any_nz |= v;
        }
        if (__syncthreads_or(any_nz)) {
#pragma unroll
            for (int r = ty; r < 32; r += 8) {
                const int x = x0 + r, y = y0 + tx;
                const int v = tile[tx][r];
                if (v && x < xw && y < yw) miss[(size_t)x * yw + y] += v;
            }
        }
        __syncthreads();  // the tile buffer is reused by the next iteration
    }
}

// ------------------------------------------------------------------------------------------
// Input screening for the host-buffer API: flags[0] |= NaN anywhere, flags[1] |= inf in oy or in a
// sensor position -- the values int() raises on in [MAP]:33-36 (inf in ox alone is legal, [MAP]:30).

template <typename CT>
__global__ void __launch_bounds__(256)
grid_validate_kernel(const CT *__restrict__ ox, const CT *__restrict__ oy, long long total,
                     const CT *__restrict__ cx, const CT *__restrict__ cy, int scans,
                     int32_t *__restrict__ flags)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    bool has_nan = false, has_inf = false;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const CT x = __ldg(ox + i), y = __ldg(oy + i);
        if (isinf(x)) continue;  // the beam is skipped before oy is looked at
        has_nan |= isnan(x) || isnan(y);
        has_inf |= isinf(y);
    }
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < scans; i += stride) {
        const CT x = __ldg(cx + i), y = __ldg(cy + i);
        has_nan |= isnan(x) || isnan(y);
        has_inf |= isinf(x) || isinf(y);
    }
    if (__any_sync(0xffffffffu, has_nan) && (threadIdx.x & 31) == 0) atomicOr(&flags[0], 1);
    if (__any_sync(0xffffffffu, has_inf) && (threadIdx.x & 31) == 0) atomicOr(&flags[1], 1);
}

// ------------------------------------------------------------------------------------------
// counts -> evidence score + occupancy (SURVEY.md section 8a row A6).  Pure streaming.

__global__ void __launch_bounds__(256)
grid_finalize_kernel(const int32_t *__restrict__ hit, const int32_t *__restrict__ miss,
                     long long cells, double w_hit, double w_miss, double thresh,
                     float *__restrict__ datamap, int8_t *__restrict__ pmap)
{
    const long long quads = cells >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += stride) {
        const int4 h = __ldg(reinterpret_cast<const int4 *>(hit) + q);
        const int4 m = __ldg(reinterpret_cast<const int4 *>(miss) + q);
        const int hh[4] = {h.x, h.y, h.z, h.w};
        const int mm[4] = {m.x, m.y, m.z, m.w};
        float sc[4];
        char pm[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double v = __dadd_rn(__dmul_rn(w_miss, (double)mm[j]), __dmul_rn(w_hit, (double)hh[j]));
            sc[j] = (float)v;
            pm[j] = (hh[j] == 0 && mm[j] == 0) ? 50 : (v > thresh ? 100 : 0);
        }
        if (datamap) reinterpret_cast<float4 *>(datamap)[q] = make_float4(sc[0], sc[1], sc[2], sc[3]);
        if (pmap) reinterpret_cast<char4 *>(pmap)[q] = make_char4(pm[0], pm[1], pm[2], pm[3]);
    }
    // tail (cells % 4)
    const long long tail0 = quads << 2;
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < cells - tail0) {
        const long long c = tail0 + g;
        const int hv = hit[c], mv = miss[c];
        const double v = __dadd_rn(__dmul_rn(w_miss, (double)mv), __dmul_rn(w_hit, (double)hv));
        if (datamap) datamap[c] = (float)v;
        if (pmap) pmap[c] = (hv == 0 && mv == 0) ? 50 : (v > thresh ? 100 : 0);
    }
}

// [SLAM]:270-271  data = pmap.T.reshape(-1): data[y * xw + x] = pmap[x][y].  32x32 smem transpose.
__global__ void __launch_bounds__(256)
grid_pack_ros_kernel(const int8_t *__restrict__ pmap, int xw, int yw, int8_t *__restrict__ data)
{
    __shared__ int8_t tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;  // bx over x, by over y
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int x = bx + r, y = by + threadIdx.x;
        if (x < xw && y < yw) tile[r][threadIdx.x] = pmap[(size_t)x * yw + y];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int y = by + r, x = bx + threadIdx.x;
        if (x < xw && y < yw) data[(size_t)y * xw + x] = tile[threadIdx.x][r];
    }
}

// [BRES]:2-58 for a batch of segments: one thread per segment writes its whole path in the
// reference's order (first cell = start, last cell = end).
__global__ void __launch_bounds__(128)
bresenham_paths_kernel(const int32_t *__restrict__ segs, int count, const int64_t *__restrict__ offsets,
                       int32_t *__restrict__ cells_xy)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    int x0 = segs[4 * i], y0 = segs[4 * i + 1], x1 = segs[4 * i + 2], y1 = segs[4 * i + 3];
    if (x0 == x1 && y0 == y1) return;
    const int steep = abs(y1 - y0) > abs(x1 - x0);
    if (steep) {
        int t = x0; x0 = y0; y0 = t;
        t = x1; x1 = y1; y1 = t;
    }
    const int flipped = x0 > x1;
    if (flipped) {
        int t = x0; x0 = x1; x1 = t;
        t = y0; y0 = y1; y1 = t;
    }
    const int span = x1 - x0;
    const double slope = __ddiv_rn((double)abs(y1 - y0), (double)span);
    const int inc = (y0 < y1) ? 1 : -1;
    int32_t *out = cells_xy + 2 * offsets[i];
    double acc = 0.0;
    int minor = y0;
    for (int k = 0; k <= span; ++k) {
        const int major = x0 + k;
        const int slot = flipped ? (span - k) : k;
        out[2 * slot] = steep ? minor : major;
        out[2 * slot + 1] = steep ? major : minor;
        bres_step(acc, minor, slope, inc);
    }
}

}  // namespace b2s

// ============================================================================== C ABI

using namespace b2s;

namespace b2s {
template <typename CT>
static int raycast_plain(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m, double off_x, double off_y,
                         const CT *ox, const CT *oy, const CT *cx, const CT *cy, int scans, int beams,
                         int32_t *counters, void *stream)
{
    B2S_REQUIRE(hit && miss && ox && oy && cx && cy, "b2s_grid_raycast: null pointer");
    B2S_REQUIRE(xw > 0 && yw > 0 && (long long)xw * yw < (1ll << 31), "b2s_grid_raycast: grid size");
    B2S_REQUIRE(scans >= 0 && beams >= 0, "b2s_grid_raycast: negative count");
    B2S_REQUIRE(cells_per_m == cells_per_m && off_x == off_x && off_y == off_y, "b2s_grid_raycast: NaN scale");
    const long long total = (long long)scans * beams;
    if (total == 0) return B2S_OK;
    const int threads = 256;
    const long long blocks = (total + threads - 1) / threads;
    B2S_REQUIRE(blocks < (1ll << 31), "b2s_grid_raycast: too many beams for one launch");
    cudaStream_t st = (cudaStream_t)stream;
    if (g_grid_variant == 1)
        grid_raycast_v1<CT><<<(unsigned)blocks, threads, 0, st>>>(hit, miss, xw, yw, cells_per_m, off_x, off_y,
                                                                  ox, oy, cx, cy, total, beams, counters);
    else if (g_grid_variant == 2)
        grid_raycast_v2<CT><<<(unsigned)blocks, threads, 0, st>>>(hit, miss, xw, yw, cells_per_m, off_x, off_y,
                                                                  ox, oy, cx, cy, total, beams, counters);
    else  // 3, and 4 without a workspace
        grid_raycast_v3<CT><<<(unsigned)blocks, threads, 0, st>>>(hit, miss, xw, yw, cells_per_m, off_x, off_y,
                                                                  ox, oy, cx, cy, total, beams, counters);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}
}  // namespace b2s

extern "C" int b2s_grid_raycast(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                                double off_x, double off_y, const float *ox, const float *oy,
                                const float *cx, const float *cy, int scans, int beams,
                                int32_t *counters, void *stream)
{
    return raycast_plain<float>(hit, miss, xw, yw, cells_per_m, off_x, off_y, ox, oy, cx, cy, scans, beams, counters,
                                stream);
}

extern "C" int b2s_grid_raycast_f64(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                                    double off_x, double off_y, const double *ox, const double *oy,
                                    const double *cx, const double *cy, int scans, int beams,
                                    int32_t *counters, void *stream)
{
    return raycast_plain<double>(hit, miss, xw, yw, cells_per_m, off_x, off_y, ox, oy, cx, cy, scans, beams, counters,
                                 stream);
}

extern "C" size_t b2s_grid_workspace_bytes(int xw, int yw)
{
    if (xw <= 0 || yw <= 0) return 0;
    return GRID_WS_HEADER + grid_dirty_bytes(xw, yw) + (size_t)xw * yw * sizeof(int32_t);
}

extern "C" int b2s_grid_workspace_init(void *workspace, int xw, int yw, void *stream)
{
    B2S_REQUIRE(workspace && xw > 0 && yw > 0, "b2s_grid_workspace_init: bad arguments");
    B2S_REQUIRE((uintptr_t)workspace % 16 == 0, "b2s_grid_workspace_init: workspace must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    B2S_CUDA(cudaMemsetAsync(workspace, 0x80, GRID_WS_HEADER, st));
    B2S_CUDA(cudaMemsetAsync((char *)workspace + GRID_WS_HEADER, 0,
                             grid_dirty_bytes(xw, yw) + (size_t)xw * yw * sizeof(int32_t), st));
    return B2S_OK;
}

namespace b2s {
// Shared by b2s_grid_raycast_ws / b2s_grid_raycast_ranges (sign +1) and the host layer's roll-back of a
// rejected batch (sign -1).
static int raycast_v4_launch(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m, double off_x,
                             double off_y, const ScanInput &in, int mode, int scans, int beams, int32_t *counters,
                             void *workspace, int sign, void *stream, bool fold)
{
    B2S_REQUIRE(hit && miss && workspace, "b2s_grid_raycast_ws: null pointer");
    B2S_REQUIRE(xw > 0 && yw > 0 && (long long)xw * yw < (1ll << 30), "b2s_grid_raycast_ws: grid size");
    B2S_REQUIRE(scans >= 0 && beams >= 0, "b2s_grid_raycast_ws: negative count");
    B2S_REQUIRE(cells_per_m == cells_per_m && off_x == off_x && off_y == off_y, "b2s_grid_raycast_ws: NaN scale");
    B2S_REQUIRE((uintptr_t)workspace % 16 == 0, "b2s_grid_raycast_ws: workspace must be 16-byte aligned");
    const long long total = (long long)scans * beams;
    if (total == 0) return B2S_OK;
    const int threads = 256;
    const long long blocks = (total + threads - 1) / threads;
    B2S_REQUIRE(blocks < (1ll << 31), "b2s_grid_raycast_ws: too many beams for one launch");
    cudaStream_t st = (cudaStream_t)stream;
    GridWorkspace *ws = (GridWorkspace *)workspace;
    uint8_t *dirty = (uint8_t *)workspace + GRID_WS_HEADER;
    int32_t *scratch_t = (int32_t *)((char *)workspace + GRID_WS_HEADER + grid_dirty_bytes(xw, yw));
#define B2S_V4(SG, FU)                                                                                             \
    do {                                                                                                           \
        if (g_grid_variant >= 5)                                                                              \
            grid_raycast_v4<SG, FU, true><<<(unsigned)blocks, threads, 0, st>>>(hit, miss, scratch_t, ws, dirty, xw, \
                                                                                 yw, cells_per_m, off_x, off_y, in,  \
                                                                                 total, beams, counters);            \
        else                                                                                                       \
            grid_raycast_v4<SG, FU, false><<<(unsigned)blocks, threads, 0, st>>>(hit, miss, scratch_t, ws, dirty,   \
                                                                                  xw, yw, cells_per_m, off_x, off_y, \
                                                                                  in, total, beams, counters);       \
    } while (0)
    // variant 6 for a batch that is applied; taking one back out stays on the variant-5 march
#define B2S_V6_LAUNCH(FU, UNITS)                                                                                   \
    do {                                                                                                           \
        const int tile_bytes = V6_TILE_WORDS * (int)sizeof(uint32_t);                                              \
        B2S_CUDA(cudaFuncSetAttribute(grid_raycast_v6<FU, UNITS>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                      tile_bytes));                                                                \
        const long long ctas = (long long)((scans + V6_SCANS - 1) / V6_SCANS) * ((beams + V6_SECTOR - 1) / V6_SECTOR); \
        B2S_REQUIRE(ctas < (1ll << 31), "b2s_grid_raycast_ws: too many beams for one launch");                  \
        grid_raycast_v6<FU, UNITS><<<(unsigned)ctas, V6_UNITS * 32 / UNITS, tile_bytes, st>>>(                     \
            hit, miss, scratch_t, ws, dirty, xw, yw, cells_per_m, off_x, off_y, in, scans, beams, counters);        \
    } while (0)
#define B2S_V6(FU)                                                                                                 \
    do {                                                                                                           \
        if (g_grid_tile_layout == 0) B2S_V6_LAUNCH(FU, 1); else B2S_V6_LAUNCH(FU, 2);                              \
    } while (0)
    if (sign >= 0 && g_grid_variant >= 6) {
        if (mode == IN_FUSED) B2S_V6(IN_FUSED); else if (mode == IN_F64) B2S_V6(IN_F64); else B2S_V6(IN_F32);
    } else if (sign >= 0) {
        if (mode == IN_FUSED) B2S_V4(1, IN_FUSED); else if (mode == IN_F64) B2S_V4(1, IN_F64); else B2S_V4(1, IN_F32);
    } else {
        if (mode == IN_FUSED) B2S_V4(-1, IN_FUSED); else if (mode == IN_F64) B2S_V4(-1, IN_F64); else B2S_V4(-1, IN_F32);
    }
#undef B2S_V4
#undef B2S_V6
#undef B2S_V6_LAUNCH
    B2S_CUDA(cudaGetLastError());
    if (!fold) return B2S_OK;
    long long ftiles = (long long)((xw + 31) / 32) * ((yw + 31) / 32);
    const long long fcap = (long long)sm_count() * 16;
    if (ftiles > fcap) ftiles = fcap;
    grid_fold_kernel<<<(unsigned)ftiles, 256, 0, st>>>(miss, scratch_t, ws, xw, yw);
    B2S_CUDA(cudaGetLastError());
    B2S_CUDA(cudaMemsetAsync(ws, 0x80, GRID_WS_HEADER, st));
    return B2S_OK;
}

int grid_raycast_signed(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m, double off_x,
                        double off_y, const void *ox, const void *oy, const void *cx, const void *cy, bool is_f64,
                        int scans, int beams, int32_t *counters, void *workspace, int sign, void *stream, bool fold)
{
    B2S_REQUIRE(ox && oy && cx && cy, "b2s_grid_raycast_ws: null pointer");
    ScanInput in = {ox, oy, cx, cy, nullptr, nullptr, nullptr, 0.0};
    return raycast_v4_launch(hit, miss, xw, yw, cells_per_m, off_x, off_y, in, is_f64 ? IN_F64 : IN_F32, scans, beams,
                             counters, workspace, sign, stream, fold);
}

int grid_raycast_ranges_signed(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m, double off_x,
                               double off_y, const float *ranges, const double *pose4, const double *beam_cs,
                               double clamp, int scans, int beams, int32_t *counters, void *workspace, int sign,
                               void *stream, bool fold)
{
    B2S_REQUIRE(ranges && pose4 && beam_cs, "b2s_grid_raycast_ranges: null pointer");
    B2S_REQUIRE((uintptr_t)pose4 % 16 == 0 && (uintptr_t)beam_cs % 16 == 0,
                "b2s_grid_raycast_ranges: pose and beam tables must be 16-byte aligned");
    ScanInput in = {nullptr, nullptr, nullptr, nullptr, ranges, pose4, beam_cs, clamp};
    return raycast_v4_launch(hit, miss, xw, yw, cells_per_m, off_x, off_y, in, IN_FUSED, scans, beams, counters,
                             workspace, sign, stream, fold);
}
}  // namespace b2s

extern "C" int b2s_grid_raycast_ranges(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                                       double off_x, double off_y, const float *ranges, const double *pose4,
                                       const double *beam_cs, double clamp_inf_to, int scans, int beams,
                                       int32_t *counters, void *workspace, void *stream)
{
    return grid_raycast_ranges_signed(hit, miss, xw, yw, cells_per_m, off_x, off_y, ranges, pose4, beam_cs,
                                      clamp_inf_to, scans, beams, counters, workspace, +1, stream);
}

extern "C" int b2s_grid_raycast_ws(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                                   double off_x, double off_y, const float *ox, const float *oy,
                                   const float *cx, const float *cy, int scans, int beams,
                                   int32_t *counters, void *workspace, void *stream)
{
    if (workspace == nullptr || g_grid_variant < 4)
        return b2s_grid_raycast(hit, miss, xw, yw, cells_per_m, off_x, off_y, ox, oy, cx, cy, scans, beams,
                                counters, stream);
    return grid_raycast_signed(hit, miss, xw, yw, cells_per_m, off_x, off_y, ox, oy, cx, cy, false, scans, beams,
                               counters, workspace, +1, stream);
}

extern "C" int b2s_grid_raycast_ws_f64(int32_t *hit, int32_t *miss, int xw, int yw, double cells_per_m,
                                       double off_x, double off_y, const double *ox, const double *oy,
                                       const double *cx, const double *cy, int scans, int beams,
                                       int32_t *counters, void *workspace, void *stream)
{
    if (workspace == nullptr || g_grid_variant < 4)
        return b2s_grid_raycast_f64(hit, miss, xw, yw, cells_per_m, off_x, off_y, ox, oy, cx, cy, scans, beams,
                                    counters, stream);
    return grid_raycast_signed(hit, miss, xw, yw, cells_per_m, off_x, off_y, ox, oy, cx, cy, true, scans, beams,
                               counters, workspace, +1, stream);
}

namespace b2s {
// Zero the tiles of `hit` / `miss` whose dirty byte is set, then clear the byte: brings a pair of delta
// planes back to all-zero at a cost proportional to what the last ray-casts touched.
__global__ void __launch_bounds__(256)
grid_clear_dirty_kernel(int32_t *__restrict__ hit, int32_t *__restrict__ miss, uint8_t *__restrict__ dirty, int xw,
                        int yw, int ntiles)
{
    const int tiles_y = grid_tiles(yw);
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {   // (fixed-size grid: a 16384^2 map has 65 536 tiles)
        if (!dirty[tile]) continue;
        const int x0 = (tile / tiles_y) * GRID_TILE, y0 = (tile % tiles_y) * GRID_TILE;
        for (int k = threadIdx.x; k < GRID_TILE * GRID_TILE; k += blockDim.x) {
            const int x = x0 + k / GRID_TILE, y = y0 + k % GRID_TILE;
            if (x < xw && y < yw) {
                const size_t at = (size_t)x * yw + y;
                hit[at] = 0;
                miss[at] = 0;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) dirty[tile] = 0;
    }
}
}  // namespace b2s

namespace b2s {
// Finalize only the dirty tiles: refresh their cells in the full device map and pack them (4096 bytes per
// tile, row-major 64 x 64) into `packed` so the host can patch its copy with a transfer proportional to
// what changed.  counter / tile_ids: number of dirty tiles and their indices (slots beyond cap are dropped;
// the caller then falls back to the full map).
__global__ void __launch_bounds__(256)
grid_finalize_dirty_kernel(const int32_t *__restrict__ hit, const int32_t *__restrict__ miss, int xw, int yw,
                           double w_hit, double w_miss, double thresh, const uint8_t *__restrict__ dirty,
                           int8_t *__restrict__ pmap, int8_t *__restrict__ packed, int32_t *__restrict__ tile_ids,
                           int32_t *__restrict__ counter, int cap, int ntiles)
{
    __shared__ int slot_s;
    const int tiles_y = grid_tiles(yw);
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {  // fixed-size grid (65 536 tiles at 16384^2)
        if (!dirty[tile]) continue;
        if (threadIdx.x == 0) slot_s = atomicAdd(counter, 1);
        __syncthreads();
        const int slot = slot_s;
        if (slot < cap && threadIdx.x == 0) tile_ids[slot] = tile;
        const int x0 = (tile / tiles_y) * GRID_TILE, y0 = (tile % tiles_y) * GRID_TILE;
        for (int k = threadIdx.x; k < GRID_TILE * GRID_TILE; k += blockDim.x) {
            const int x = x0 + k / GRID_TILE, y = y0 + k % GRID_TILE;
            int8_t v = 0;
            if (x < xw && y < yw) {
                const size_t at = (size_t)x * yw + y;
                const int h = hit[at], m = miss[at];
                const double sc = __dadd_rn(__dmul_rn(w_miss, (double)m), __dmul_rn(w_hit, (double)h));
                v = (h == 0 && m == 0) ? 50 : (sc > thresh ? 100 : 0);
                pmap[at] = v;
            }
            if (slot < cap) packed[(size_t)slot * GRID_TILE * GRID_TILE + k] = v;
        }
        __syncthreads();  // slot_s is rewritten by the next dirty tile of this CTA
    }
}

int grid_finalize_dirty(const int32_t *hit, const int32_t *miss, int xw, int yw, double w_hit, double w_miss,
                        double thresh, void *workspace, int8_t *pmap, int8_t *packed, int32_t *tile_ids,
                        int32_t *counter, int cap, void *stream)
{
    const int tiles = grid_tiles(xw) * grid_tiles(yw);
    const int gcap = sm_count() * 16;
    grid_finalize_dirty_kernel<<<tiles < gcap ? tiles : gcap, 256, 0, (cudaStream_t)stream>>>(
        hit, miss, xw, yw, w_hit, w_miss, thresh, (const uint8_t *)workspace + GRID_WS_HEADER, pmap, packed, tile_ids,
        counter, cap, tiles);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}
}  // namespace b2s

extern "C" void *b2s_grid_workspace_dirty(void *workspace)
{
    return workspace ? (void *)((char *)workspace + GRID_WS_HEADER) : nullptr;
}

extern "C" int b2s_grid_tile_count(int xw, int yw, int *tiles_x, int *tiles_y)
{
    B2S_REQUIRE(xw > 0 && yw > 0, "b2s_grid_tile_count: grid size");
    if (tiles_x) *tiles_x = grid_tiles(xw);
    if (tiles_y) *tiles_y = grid_tiles(yw);
    return B2S_OK;
}

extern "C" int b2s_grid_clear_dirty(int32_t *hit, int32_t *miss, int xw, int yw, void *workspace, void *stream)
{
    B2S_REQUIRE(hit && miss && workspace && xw > 0 && yw > 0, "b2s_grid_clear_dirty: bad arguments");
    const int tiles = grid_tiles(xw) * grid_tiles(yw);
    const int cap = sm_count() * 16;
    grid_clear_dirty_kernel<<<tiles < cap ? tiles : cap, 256, 0, (cudaStream_t)stream>>>(
        hit, miss, (uint8_t *)workspace + GRID_WS_HEADER, xw, yw, tiles);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

namespace b2s {
template <typename CT>
static int validate_impl(const CT *ox, const CT *oy, const CT *cx, const CT *cy, int scans, int beams, int32_t *flags,
                         void *stream)
{
    B2S_REQUIRE(scans >= 0 && beams >= 0, "b2s_grid_validate: negative count");
    B2S_REQUIRE(flags, "b2s_grid_validate: null flags");
    if (scans == 0) return B2S_OK;
    B2S_REQUIRE(cx && cy && (beams == 0 || (ox && oy)), "b2s_grid_validate: null pointer");
    const long long total = (long long)scans * beams;
    long long blocks = (total + 256 * 8 - 1) / (256 * 8);
    const long long cap = (long long)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    grid_validate_kernel<CT><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(ox, oy, total, cx, cy, scans, flags);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}
}  // namespace b2s

extern "C" int b2s_grid_validate(const float *ox, const float *oy, const float *cx, const float *cy,
                                 int scans, int beams, int32_t *flags, void *stream)
{
    return validate_impl<float>(ox, oy, cx, cy, scans, beams, flags, stream);
}

extern "C" int b2s_grid_validate_f64(const double *ox, const double *oy, const double *cx, const double *cy,
                                     int scans, int beams, int32_t *flags, void *stream)
{
    return validate_impl<double>(ox, oy, cx, cy, scans, beams, flags, stream);
}

extern "C" int b2s_grid_finalize(const int32_t *hit, const int32_t *miss, int xw, int yw, double w_hit,
                                 double w_miss, double thresh, float *datamap, int8_t *pmap,
                                 void *stream)
{
    B2S_REQUIRE(hit && miss, "b2s_grid_finalize: null plane");
    B2S_REQUIRE(xw > 0 && yw > 0, "b2s_grid_finalize: grid size");
    if (!datamap && !pmap) return B2S_OK;
    const long long cells = (long long)xw * yw;
    B2S_REQUIRE(((uintptr_t)hit % 16 == 0) && ((uintptr_t)miss % 16 == 0) &&
                    (!datamap || (uintptr_t)datamap % 16 == 0) && (!pmap || (uintptr_t)pmap % 4 == 0),
                "b2s_grid_finalize: planes must be 16-byte aligned");
    const int threads = 256;
    long long want = ((cells >> 2) + threads - 1) / threads;
    const long long cap = (long long)sm_count() * 16;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    grid_finalize_kernel<<<(unsigned)want, threads, 0, (cudaStream_t)stream>>>(hit, miss, cells, w_hit, w_miss,
                                                                              thresh, datamap, pmap);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

extern "C" int b2s_grid_pack_ros(const int8_t *pmap, int xw, int yw, int8_t *data, void *stream)
{
    B2S_REQUIRE(pmap && data, "b2s_grid_pack_ros: null pointer");
    B2S_REQUIRE(xw > 0 && yw > 0, "b2s_grid_pack_ros: grid size");
    dim3 grid((xw + 31) / 32, (yw + 31) / 32), block(32, 8);
    grid_pack_ros_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(pmap, xw, yw, data);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}

extern "C" int b2s_bresenham_paths(const int32_t *segs, int count, const int64_t *offsets,
                                   int32_t *cells_xy, void *stream)
{
    B2S_REQUIRE(count >= 0, "b2s_bresenham_paths: negative count");
    if (count == 0) return B2S_OK;
    B2S_REQUIRE(segs && offsets && cells_xy, "b2s_bresenham_paths: null pointer");
    bresenham_paths_kernel<<<(count + 127) / 128, 128, 0, (cudaStream_t)stream>>>(segs, count, offsets, cells_xy);
    B2S_CUDA(cudaGetLastError());
    return B2S_OK;
}
