// Layer 2 of the C ABI: host-buffer entry points (the calls the Python ICP / Mapping classes
// make), error reporting, and NCCL plumbing for the count-delta all-reduce.
#include "b2s_common.cuh"

#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <new>

namespace b2s {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int sm_count()
{
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

extern int g_grid_variant;
extern int g_grid_tile_layout;
extern int g_icp_src_per_thread;
extern int g_icp_prune;
extern int g_icp_block;
extern int g_icp_layout;
int g_icp_graph = 1;  // 1: single-pair ICP calls replay a captured CUDA graph (default); 0: plain stream calls (tuning hook)
constexpr int MAX_CHUNKS = 16;
int g_tune_gen = 0;    // bumped by every b2s_tune: cached single-pair graphs captured under other settings are stale
int g_h2d_chunks = 0;  // 0: automatic; 1..MAX_CHUNKS force the pipeline depth of the host-buffer calls (tuning hook)

// Pipeline depth of a host-buffer call: the call's own measured choice `want`, at most `cap`, unless h2d_chunks forces
// one; never more chunks than there are units (pairs, scans) to cut, never fewer than one.
static int pipeline_chunks(int want, int cap, int units)
{
    int n = want < cap ? want : cap;
    if (g_h2d_chunks > 0) n = g_h2d_chunks;
    if (n > units) n = units;
    return n < 1 ? 1 : n;
}

ScratchPool *scratch_pool()
{
    static thread_local ScratchPool *pool = nullptr;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    if (!pool) pool = new (std::nothrow) ScratchPool();
    if (!pool) return nullptr;
    if (pool->device != dev) {  // the thread moved to another GPU: its buffers live on the old one
        if (pool->device >= 0 && cudaSetDevice(pool->device) == cudaSuccess) {
            pool->a.release();
            pool->b.release();
            pool->c.release();
            cudaSetDevice(dev);
        }
        pool->a = Buf();
        pool->b = Buf();
        pool->c = Buf();
        pool->device = dev;
    }
    return pool;
}

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (dev >= 0 && dev != prev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// Timeline of one host-buffer call, printed to stderr when B2S_TRACE is set in the environment: CUDA events on
// the copy and compute streams (ms since the call started on the device) and host timestamps (ms since entry).
// Diagnostic only; with the variable unset it costs one getenv per call.
struct Trace {
    struct Mark {
        const char *what;
        int k;
        cudaEvent_t ev;
        double host_ms;
    };
    bool on = false;
    int n = 0;
    Mark marks[96];
    cudaEvent_t t0 = nullptr;
    timespec h0;
    explicit Trace(cudaStream_t s)
    {
        on = getenv("B2S_TRACE") != nullptr;
        if (!on) return;
        clock_gettime(CLOCK_MONOTONIC, &h0);
        if (cudaEventCreate(&t0) != cudaSuccess || cudaEventRecord(t0, s) != cudaSuccess) on = false;
    }
    double host_now() const
    {
        timespec t;
        clock_gettime(CLOCK_MONOTONIC, &t);
        return (t.tv_sec - h0.tv_sec) * 1e3 + (t.tv_nsec - h0.tv_nsec) * 1e-6;
    }
    void mark(const char *what, int k, cudaStream_t s)  // s == nullptr: host-only mark
    {
        if (!on || n >= 96) return;
        Mark &m = marks[n];
        m.what = what;
        m.k = k;
        m.ev = nullptr;
        m.host_ms = host_now();
        if (s && (cudaEventCreate(&m.ev) != cudaSuccess || cudaEventRecord(m.ev, s) != cudaSuccess)) m.ev = nullptr;
        ++n;
    }
    ~Trace()
    {
        if (!on) return;
        cudaDeviceSynchronize();
        fprintf(stderr, "[b2s trace] %-28s %10s %10s\n", "mark", "device ms", "host ms");
        for (int i = 0; i < n; ++i) {
            float ms = -1.0f;
            if (marks[i].ev) {
                cudaEventElapsedTime(&ms, t0, marks[i].ev);
                cudaEventDestroy(marks[i].ev);
            }
            fprintf(stderr, "[b2s trace] %-24s %3d %10.3f %10.3f\n", marks[i].what, marks[i].k, ms, marks[i].host_ms);
        }
        fprintf(stderr, "[b2s trace] %-28s %10s %10.3f\n", "return", "", host_now());
        cudaEventDestroy(t0);
    }
};

// The streams and events of an object's chunked pipeline, shared by ICP and Mapping.  stream: everything ordered and
// the blocking calls' read-back; stream2: every other chunk's compute, so that the ragged end of one chunk (ICP pairs
// need 2..max_iter iterations, beams differ in length) overlaps the next chunk instead of idling the device;
// copy_stream: H2D, chunk k followed by chunk_ready[k]; d2h_stream: the streaming calls' read-back, after `handoff` on
// stream.  Slot: one streaming call in flight, with inputs_free (its inputs may be overwritten) and done (its
// results are on the host).
template <class Slot>
struct StreamSet {
    cudaStream_t stream = nullptr, stream2 = nullptr, copy_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t chunk_ready[MAX_CHUNKS] = {}, joined = nullptr, handoff = nullptr;
    Slot slot[2];

    cudaError_t create()
    {
        cudaStream_t *streams[] = {&stream, &stream2, &copy_stream, &d2h_stream};
        cudaEvent_t *events[] = {&joined, &handoff, &slot[0].inputs_free, &slot[0].done, &slot[1].inputs_free, &slot[1].done};
        cudaError_t e = cudaSuccess;
        for (cudaStream_t *s : streams)
            if (e == cudaSuccess) e = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking);
        for (cudaEvent_t *ev : events)
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
        for (cudaEvent_t &ev : chunk_ready)
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
        return e;
    }
    // Waits for all four streams, lets the owner free its buffers, then destroys the handles.
    template <class FreeBuffers>
    void teardown(FreeBuffers free_buffers)
    {
        cudaStream_t streams[] = {stream, stream2, copy_stream, d2h_stream};
        for (cudaStream_t s : streams)
            if (s) cudaStreamSynchronize(s);
        free_buffers();
        cudaEvent_t events[] = {joined, handoff, slot[0].inputs_free, slot[0].done, slot[1].inputs_free, slot[1].done};
        for (cudaEvent_t ev : events)
            if (ev) cudaEventDestroy(ev);
        for (cudaEvent_t ev : chunk_ready)
            if (ev) cudaEventDestroy(ev);
        for (cudaStream_t s : streams)
            if (s) cudaStreamDestroy(s);
    }
};

}  // namespace b2s

using namespace b2s;

// Streaming sequence calls (b2s_icp_submit_sequence / _scans, b2s_icp_wait): two slots of device buffers, so the
// scans of call k + 1 cross PCIe while call k is being solved and its transforms are read back.
struct IcpSlot {
    Buf d_scans, d_T, d_iters, d_cs;
    cudaEvent_t inputs_free = nullptr, done = nullptr;
    bool in_flight = false;
    int ticket = 0;
};

struct b2s_icp : StreamSet<IcpSlot> {
    int device = 0;
    Buf d_tar, d_src, d_T, d_iters, d_aux;
    // The per-scan call of the ROS node (ICP.process: ONE pair) is launch-bound, so its device work -- two uploads,
    // the solve, two read-backs -- is captured once into a CUDA graph and replayed with one launch.  The graph is
    // tied to the sizes, parameters and buffer addresses below and re-captured when any of them changes.
    Buf h_one = {nullptr, 0, true};  // pinned staging: [tar][src][T (9 doubles)][iterations]
    cudaGraphExec_t one_exec = nullptr;
    struct {
        int is_f64, n_src, n_tar, max_iter, tune_gen;
        double tol;
        void *d_tar, *d_src, *d_T, *d_iters, *h;
    } one_key = {};
    int submitted = 0;
    // Map observation (b2s_icp_set_map / b2s_icp_map_observation): the static map obs_x | obs_y, kept until replaced;
    // the call's uploads (beam table | poses | ranges), and the target (+ virtual ranges) and source clouds it builds.
    Buf d_map, d_map_in, d_map_tar, d_map_src;
    int map_count = 0;
};

namespace {
// One host batch in either input form.
struct HostBatch {
    bool fused;
    bool f64;                        // endpoints form: float64 (the reference's dtype) instead of float32
    const void *ox, *oy, *cx, *cy;   // endpoints form
    const float *ranges;             // fused form
    const double *pose4, *beam_cs;   // pose4 [scans][4] = x, y, cos yaw, sin yaw ...
    double clamp;
    const double *poses3;            // ... or poses3 [scans][3] = x, y, yaw: the table is built here, chunk by chunk
};

// The same batch in one device buffer: ox | oy | cx | cy, or ranges | pose table [scans][4] | beam table [beams][2],
// each region 16-byte aligned.  A streamed step keeps its DeviceBatch until its wait, so a rejected step is taken
// back out of exactly the bytes it was ray-cast from.
struct DeviceBatch {
    bool fused = false, f64 = false;
    int scans = 0, beams = 0;
    double clamp = 0.0;
    char *pts = nullptr, *oy = nullptr, *cx = nullptr, *cy = nullptr;  // pts: ox, or the ranges
    double *pose = nullptr, *cs = nullptr;

    DeviceBatch() = default;
    DeviceBatch(const HostBatch &hb, int scans, int beams)
        : fused(hb.fused), f64(!hb.fused && hb.f64), scans(scans), beams(beams), clamp(hb.clamp) {}
    size_t el() const { return f64 ? sizeof(double) : sizeof(float); }  // bytes per input coordinate
    size_t a_pts() const { return ((size_t)scans * beams * el() + 15) & ~(size_t)15; }
    size_t a_ctr() const { return ((size_t)scans * el() + 15) & ~(size_t)15; }
    size_t bytes() const
    {
        return fused ? a_pts() + (size_t)scans * 4 * sizeof(double) + (size_t)beams * 2 * sizeof(double)
                     : 2 * a_pts() + 2 * a_ctr();
    }
    void bind(void *base)
    {
        pts = (char *)base;
        oy = pts + a_pts();
        cx = oy + a_pts();
        cy = cx + a_ctr();
        pose = (double *)oy;
        cs = pose + (size_t)scans * 4;
    }
    // Copies scans [s0, s1) of hb on stream st; the first chunk also brings the beam table.  With hb.poses3 the rows
    // [s0, s1) of the pinned pose_table are computed first: the host runs ahead of the device, so the table of chunk
    // k + 1 (u2T's math.cos / math.sin, [SLAM]:130-137: the same libm calls) is made while chunk k crosses PCIe.
    int upload(const HostBatch &hb, size_t s0, size_t s1, double *pose_table, cudaStream_t st) const
    {
        const size_t ns = s1 - s0;
        if (!fused) {
            const size_t e = el();
            B2S_CUDA(cudaMemcpyAsync(pts + s0 * beams * e, (const char *)hb.ox + s0 * beams * e, ns * beams * e, cudaMemcpyHostToDevice, st));
            B2S_CUDA(cudaMemcpyAsync(oy + s0 * beams * e, (const char *)hb.oy + s0 * beams * e, ns * beams * e, cudaMemcpyHostToDevice, st));
            B2S_CUDA(cudaMemcpyAsync(cx + s0 * e, (const char *)hb.cx + s0 * e, ns * e, cudaMemcpyHostToDevice, st));
            B2S_CUDA(cudaMemcpyAsync(cy + s0 * e, (const char *)hb.cy + s0 * e, ns * e, cudaMemcpyHostToDevice, st));
            return B2S_OK;
        }
        if (s0 == 0) B2S_CUDA(cudaMemcpyAsync(cs, hb.beam_cs, (size_t)beams * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
        const double *pose4 = hb.pose4;
        if (hb.poses3) {
            for (size_t s = s0; s < s1; ++s) {
                pose_table[4 * s] = hb.poses3[3 * s];
                pose_table[4 * s + 1] = hb.poses3[3 * s + 1];
                pose_table[4 * s + 2] = cos(hb.poses3[3 * s + 2]);
                pose_table[4 * s + 3] = sin(hb.poses3[3 * s + 2]);
            }
            pose4 = pose_table;
        }
        B2S_CUDA(cudaMemcpyAsync((float *)pts + s0 * beams, hb.ranges + s0 * beams, ns * beams * sizeof(float), cudaMemcpyHostToDevice, st));
        B2S_CUDA(cudaMemcpyAsync(pose + 4 * s0, pose4 + 4 * s0, ns * 4 * sizeof(double), cudaMemcpyHostToDevice, st));
        return B2S_OK;
    }
    // Ray-casts scans [s0, s1) into m's counts with the given sign; fold: the last launch of the batch
    int raycast(const b2s_mapping *m, size_t s0, size_t s1, int sign, int32_t *counters, cudaStream_t st, bool fold) const;
};
}  // namespace

// Streaming calls (b2s_mapping_submit* / b2s_mapping_wait): two slots of everything a step owns, so that step k + 1
// can be uploaded and ray-cast while the map of step k is still on its way back to the host.
struct MappingSlot {
    Buf d_in, d_map, h_pose = {nullptr, 0, true};  // device inputs, device copy of this step's occupancy, pinned pose table
    int32_t *d_cnt = nullptr, *h_cnt = nullptr;     // the ray-cast's B2S_CNT_* words of this step (device / pinned host)
    cudaEvent_t inputs_free = nullptr, done = nullptr;  // last ray-cast of the step enqueued / results on the host
    bool in_flight = false;
    int ticket = 0;
    DeviceBatch batch;                              // the step's inputs in d_in
};

// stream carries the zeroing, the last chunk with its fold, the finalize and the blocking read-back.
struct b2s_mapping : StreamSet<MappingSlot> {
    int device;
    int xw, yw;
    double xyreso, cells_per_m, off_x, off_y;
    double w_hit, w_miss, thresh;
    cudaEvent_t begun = nullptr;
    int32_t *hit = nullptr, *miss = nullptr;
    int32_t *counters = nullptr;
    void *workspace = nullptr;
    Buf d_in, d_datamap, d_pmap, d_packed;
    Buf h_pose = {nullptr, 0, true};  // pinned [scans][4] pose table of the call in flight (b2s_mapping_update_scans)
    bool pmap_valid = false;  // d_pmap holds the occupancy of the current counts
    int8_t *h_packed = nullptr;  // pinned staging for the dirty tiles
    int32_t *h_ids = nullptr;
    int submitted = 0;
};

int DeviceBatch::raycast(const b2s_mapping *m, size_t s0, size_t s1, int sign, int32_t *counters, cudaStream_t st,
                         bool fold) const
{
    if (fused)
        return grid_raycast_ranges_signed(m->hit, m->miss, m->xw, m->yw, m->cells_per_m, m->off_x, m->off_y,
                                          (const float *)pts + s0 * beams, pose + 4 * s0, cs, clamp, (int)(s1 - s0), beams,
                                          counters, m->workspace, sign, st, fold);
    return grid_raycast_signed(m->hit, m->miss, m->xw, m->yw, m->cells_per_m, m->off_x, m->off_y, pts + s0 * beams * el(),
                               oy + s0 * beams * el(), cx + s0 * el(), cy + s0 * el(), f64, (int)(s1 - s0), beams, counters,
                               m->workspace, sign, st, fold);
}

extern "C" int b2s_version(void) { return 100; }

extern "C" const char *b2s_status_string(int status)
{
    switch (status) {
    case B2S_OK: return "ok";
    case B2S_ERR_INVALID_ARG: return "invalid argument";
    case B2S_ERR_NONFINITE: return "non-finite coordinate";
    case B2S_ERR_CUDA: return "CUDA error";
    case B2S_ERR_TOO_LONG: return "beam longer than B2S_MAX_PATH_CELLS";
    case B2S_ERR_NCCL: return "NCCL error";
    case B2S_ERR_NOMEM: return "out of memory";
    default: return "unknown status";
    }
}

extern "C" const char *b2s_last_error(void) { return g_err; }

extern "C" int b2s_device_count(int *count)
{
    B2S_REQUIRE(count, "b2s_device_count: null pointer");
    *count = 0;
    B2S_CUDA(cudaGetDeviceCount(count));
    return B2S_OK;
}

// Tuning hook used by bench.py to compare kernel variants; not part of the reference surface.
extern "C" int b2s_tune(const char *key, int value)
{
    B2S_REQUIRE(key, "b2s_tune: null key");
    ++g_tune_gen;
    if (strcmp(key, "grid_variant") == 0) {
        B2S_REQUIRE(value >= 1 && value <= 6, "b2s_tune: grid_variant must be 1..6");
        g_grid_variant = value;
        return B2S_OK;
    }
    if (strcmp(key, "grid_tile_layout") == 0) {
        B2S_REQUIRE(value == 0 || value == 1, "b2s_tune: grid_tile_layout must be 0 or 1");
        g_grid_tile_layout = value;
        return B2S_OK;
    }
    if (strcmp(key, "h2d_chunks") == 0) {
        B2S_REQUIRE(value >= 0 && value <= MAX_CHUNKS, "b2s_tune: h2d_chunks must be 0..16");
        g_h2d_chunks = value;
        return B2S_OK;
    }
    if (strcmp(key, "icp_block") == 0) {
        B2S_REQUIRE(value == 0 || value == 8 || value == 16 || value == 32, "b2s_tune: icp_block must be 0, 8, 16 or 32");
        g_icp_block = value;
        return B2S_OK;
    }
    if (strcmp(key, "icp_graph") == 0) {
        B2S_REQUIRE(value == 0 || value == 1, "b2s_tune: icp_graph must be 0 or 1");
        g_icp_graph = value;
        return B2S_OK;
    }
    if (strcmp(key, "icp_layout") == 0) {
        B2S_REQUIRE(value >= 0 && value <= 2, "b2s_tune: icp_layout must be 0, 1 or 2");
        g_icp_layout = value;
        return B2S_OK;
    }
    if (strcmp(key, "icp_prune") == 0) {
        B2S_REQUIRE(value >= 0 && value <= 4, "b2s_tune: icp_prune must be 0..4");
        g_icp_prune = value;
        return B2S_OK;
    }
    if (strcmp(key, "icp_src_per_thread") == 0) {
        B2S_REQUIRE(value == 0 || (value >= 2 && value <= 4), "b2s_tune: icp_src_per_thread must be 0, 2, 3 or 4");
        g_icp_src_per_thread = value;
        return B2S_OK;
    }
    set_error("b2s_tune: unknown key %s", key);
    return B2S_ERR_INVALID_ARG;
}

// Page-locked host memory for callers without their own allocator (Mapping's result buffer).
extern "C" int b2s_host_alloc(void **out, size_t bytes)
{
    B2S_REQUIRE(out, "b2s_host_alloc: null pointer");
    *out = nullptr;
    cudaError_t e = cudaMallocHost(out, bytes ? bytes : 1);
    if (e != cudaSuccess) {
        *out = nullptr;
        cuda_fail(e, "cudaMallocHost");
        return e == cudaErrorMemoryAllocation ? B2S_ERR_NOMEM : B2S_ERR_CUDA;
    }
    return B2S_OK;
}

extern "C" int b2s_host_free(void *p)
{
    if (p) B2S_CUDA(cudaFreeHost(p));
    return B2S_OK;
}

// ------------------------------------------------------------------------------ ICP object

extern "C" int b2s_icp_create(b2s_icp **out, int device)
{
    B2S_REQUIRE(out, "b2s_icp_create: null pointer");
    *out = nullptr;
    int ndev = 0;
    B2S_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev <= 0) {
        set_error("no CUDA device");
        return B2S_ERR_CUDA;
    }
    if (device < 0) B2S_CUDA(cudaGetDevice(&device));
    B2S_REQUIRE(device < ndev, "b2s_icp_create: device index out of range");
    DeviceGuard g(device);
    b2s_icp *c = new (std::nothrow) b2s_icp();
    if (!c) return B2S_ERR_NOMEM;
    c->device = device;
    cudaError_t e = c->create();
    if (e != cudaSuccess) {
        int rc = cuda_fail(e, "b2s_icp_create");
        b2s_icp_destroy(c);
        return rc;
    }
    *out = c;
    return B2S_OK;
}

extern "C" int b2s_icp_destroy(b2s_icp *c)
{
    if (!c) return B2S_OK;
    DeviceGuard g(c->device);
    c->teardown([c] {
        if (c->one_exec) cudaGraphExecDestroy(c->one_exec);
        c->d_tar.release(); c->d_src.release(); c->d_T.release(); c->d_iters.release(); c->d_aux.release();
        c->h_one.release();
        for (IcpSlot &sl : c->slot) {
            sl.d_scans.release(); sl.d_T.release(); sl.d_iters.release(); sl.d_cs.release();
        }
        c->d_map.release(); c->d_map_in.release(); c->d_map_tar.release(); c->d_map_src.release();
    });
    delete c;
    return B2S_OK;
}

// ICP.process for ONE pair through the captured graph (see b2s_icp::one_exec).
static int icp_process_one_graph(b2s_icp *c, const void *tar_xy, const void *src_xy, int is_f64, int n_src, int n_tar,
                                 int max_iter, double tol, double *T_out, int32_t *iters_out)
{
    const size_t el = is_f64 ? 8 : 4;
    const size_t tb = ((size_t)2 * n_tar * el + 15) & ~(size_t)15, sb = ((size_t)2 * n_src * el + 15) & ~(size_t)15;
    int rc;
    if ((rc = c->d_tar.reserve(tb))) return rc;
    if ((rc = c->d_src.reserve(sb))) return rc;
    if ((rc = c->d_T.reserve(9 * sizeof(double)))) return rc;
    if ((rc = c->d_iters.reserve(sizeof(int32_t)))) return rc;
    if ((rc = c->h_one.reserve(tb + sb + 9 * sizeof(double) + 16))) return rc;
    char *h_tar = (char *)c->h_one.p, *h_src = h_tar + tb;
    double *h_T = (double *)(h_src + sb);
    int32_t *h_it = (int32_t *)(h_T + 9);
    memcpy(h_tar, tar_xy, (size_t)2 * n_tar * el);
    memcpy(h_src, src_xy, (size_t)2 * n_src * el);
    auto &k = c->one_key;
    const bool hit = c->one_exec && k.tune_gen == g_tune_gen && k.is_f64 == is_f64 && k.n_src == n_src && k.n_tar == n_tar && k.max_iter == max_iter &&
                     k.tol == tol && k.d_tar == c->d_tar.p && k.d_src == c->d_src.p && k.d_T == c->d_T.p &&
                     k.d_iters == c->d_iters.p && k.h == c->h_one.p;
    if (!hit) {
        if (c->one_exec) {
            cudaGraphExecDestroy(c->one_exec);
            c->one_exec = nullptr;
        }
        cudaGraph_t graph = nullptr;
        B2S_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        cudaError_t e = cudaMemcpyAsync(c->d_tar.p, h_tar, (size_t)2 * n_tar * el, cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_src.p, h_src, (size_t)2 * n_src * el, cudaMemcpyHostToDevice, c->stream);
        rc = B2S_OK;
        if (e == cudaSuccess)
            rc = is_f64 ? b2s_icp_batch_f64((const double *)c->d_tar.p, (const double *)c->d_src.p, 1, n_src, n_tar, max_iter, tol,
                                            (double *)c->d_T.p, (int32_t *)c->d_iters.p, c->stream)
                        : b2s_icp_batch_f32((const float *)c->d_tar.p, (const float *)c->d_src.p, 1, n_src, n_tar, max_iter, tol,
                                            (double *)c->d_T.p, (int32_t *)c->d_iters.p, c->stream);
        if (e == cudaSuccess && rc == B2S_OK)
            e = cudaMemcpyAsync(h_T, c->d_T.p, 9 * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess && rc == B2S_OK)
            e = cudaMemcpyAsync(h_it, c->d_iters.p, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream);
        const cudaError_t e_end = cudaStreamEndCapture(c->stream, &graph);  // always leave capture mode
        if (rc != B2S_OK || e != cudaSuccess || e_end != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            if (rc != B2S_OK) return rc;  // argument errors keep their message (b2s_icp_batch: ...)
            return cuda_fail(e != cudaSuccess ? e : e_end, "b2s_icp_process: graph capture");
        }
        e = cudaGraphInstantiate(&c->one_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) {
            c->one_exec = nullptr;
            return cuda_fail(e, "b2s_icp_process: cudaGraphInstantiate");
        }
        k.tune_gen = g_tune_gen;
        k.is_f64 = is_f64; k.n_src = n_src; k.n_tar = n_tar; k.max_iter = max_iter; k.tol = tol;
        k.d_tar = c->d_tar.p; k.d_src = c->d_src.p; k.d_T = c->d_T.p; k.d_iters = c->d_iters.p; k.h = c->h_one.p;
    }
    B2S_CUDA(cudaGraphLaunch(c->one_exec, c->stream));
    B2S_CUDA(cudaStreamSynchronize(c->stream));
    memcpy(T_out, h_T, 9 * sizeof(double));
    if (iters_out) *iters_out = *h_it;
    return B2S_OK;
}

// The chunked pipeline of the ICP calls: `units` (pairs or scans) cut into nchunk chunks.  All uploads
// upload(k, u0, u1, stream) of chunks k = [u0, u1) are enqueued on the copy stream first, so that chunk k + 1 crosses
// PCIe while chunk k is solved; then solve(k, u0, u1, stream) of each chunk, alternating between stream and stream2.
// Everything after it (read-back, pose chain) is ordered on c->stream.
template <class Upload, class Solve>
static int icp_pipeline(b2s_icp *c, Trace &tr, int units, int nchunk, Upload upload, Solve solve)
{
    int rc;
    for (int k = 0; k < nchunk; ++k) {
        if ((rc = upload(k, (size_t)units * k / nchunk, (size_t)units * (k + 1) / nchunk, c->copy_stream))) return rc;
        B2S_CUDA(cudaEventRecord(c->chunk_ready[k], c->copy_stream));
        tr.mark("h2d chunk done", k, c->copy_stream);
    }
    for (int k = 0; k < nchunk; ++k) {
        cudaStream_t ks = (k & 1) ? c->stream2 : c->stream;
        B2S_CUDA(cudaStreamWaitEvent(ks, c->chunk_ready[k], 0));
        if ((rc = solve(k, (size_t)units * k / nchunk, (size_t)units * (k + 1) / nchunk, ks))) return rc;
        tr.mark("icp chunk done", k, ks);
    }
    if (nchunk > 1) {
        B2S_CUDA(cudaEventRecord(c->joined, c->stream2));
        B2S_CUDA(cudaStreamWaitEvent(c->stream, c->joined, 0));
    }
    return B2S_OK;
}

// The ending of the blocking ICP calls: the transforms and iteration counts of `pairs` pairs from c->d_T / c->d_iters
// (T_out / iters_out may be NULL), then the synchronize of c->stream.
static int icp_read_back(b2s_icp *c, Trace &tr, int pairs, double *T_out, int32_t *iters_out)
{
    if (T_out && pairs > 0)
        B2S_CUDA(cudaMemcpyAsync(T_out, c->d_T.p, (size_t)pairs * 9 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (iters_out && pairs > 0)
        B2S_CUDA(cudaMemcpyAsync(iters_out, c->d_iters.p, (size_t)pairs * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                 c->stream));
    tr.mark("results d2h done", 0, c->stream);
    B2S_CUDA(cudaStreamSynchronize(c->stream));
    tr.mark("synchronized", 0, nullptr);
    return B2S_OK;
}

extern "C" int b2s_icp_process(b2s_icp *c, const void *tar_xy, const void *src_xy, int is_f64,
                               int pairs, int n_src, int n_tar, int max_iter, double tol,
                               double *T_out, int32_t *iters_out)
{
    B2S_REQUIRE(c, "b2s_icp_process: null handle");
    B2S_REQUIRE(pairs >= 0 && n_src > 0 && n_tar > 0 && max_iter >= 0, "b2s_icp_process: bad sizes");
    if (pairs == 0) return B2S_OK;
    B2S_REQUIRE(tar_xy && src_xy && T_out, "b2s_icp_process: null pointer");
    DeviceGuard g(c->device);
    if (pairs == 1 && g_icp_graph && !getenv("B2S_TRACE"))
        return icp_process_one_graph(c, tar_xy, src_xy, is_f64, n_src, n_tar, max_iter, tol, T_out, iters_out);
    Trace tr(c->stream);
    const size_t el = is_f64 ? 8 : 4;
    const size_t tb = (size_t)pairs * 2 * n_tar * el, sb = (size_t)pairs * 2 * n_src * el;
    int rc;
    if ((rc = c->d_tar.reserve(tb))) return rc;
    if ((rc = c->d_src.reserve(sb))) return rc;
    if ((rc = c->d_T.reserve((size_t)pairs * 9 * sizeof(double)))) return rc;
    if ((rc = c->d_iters.reserve((size_t)pairs * sizeof(int32_t)))) return rc;
    const int nchunk = pipeline_chunks((int)((tb + sb + (16u << 20) - 1) / (16u << 20)), 8, pairs);  // ~16 MB of points per chunk (measured best)
    const size_t tpair = (size_t)2 * n_tar * el, spair = (size_t)2 * n_src * el;
    char *d_tar = (char *)c->d_tar.p, *d_src = (char *)c->d_src.p;
    // (every call ends with a synchronize, so the device input buffers are free to overwrite here)
    auto upload = [&](int, size_t p0, size_t p1, cudaStream_t st) -> int {
        B2S_CUDA(cudaMemcpyAsync(d_tar + p0 * tpair, (const char *)tar_xy + p0 * tpair, (p1 - p0) * tpair,
                                 cudaMemcpyHostToDevice, st));
        B2S_CUDA(cudaMemcpyAsync(d_src + p0 * spair, (const char *)src_xy + p0 * spair, (p1 - p0) * spair,
                                 cudaMemcpyHostToDevice, st));
        return B2S_OK;
    };
    auto solve = [&](int, size_t p0, size_t p1, cudaStream_t ks) {
        double *dT = (double *)c->d_T.p + p0 * 9;
        int32_t *dI = (int32_t *)c->d_iters.p + p0;
        if (is_f64)
            return b2s_icp_batch_f64((const double *)(d_tar + p0 * tpair), (const double *)(d_src + p0 * spair), (int)(p1 - p0),
                                     n_src, n_tar, max_iter, tol, dT, dI, ks);
        return b2s_icp_batch_f32((const float *)(d_tar + p0 * tpair), (const float *)(d_src + p0 * spair), (int)(p1 - p0),
                                 n_src, n_tar, max_iter, tol, dT, dI, ks);
    };
    if ((rc = icp_pipeline(c, tr, pairs, nchunk, upload, solve))) return rc;
    return icp_read_back(c, tr, pairs, T_out, iters_out);
}

// LiDAR odometry over a scan sequence ([LOC9]:159-168, [SLAM]:109-113: the target of pair k is scan k, the source
// is scan k + 1).  Every scan crosses PCIe ONCE (the pair form ships each scan twice) and the kernel reads the
// pairs in place: tar = scans, src = scans + one scan, same pair stride.  Enqueues copies and kernels only; the
// results stay in c->d_T / c->d_iters for the caller to read back or chain.
// `beam_cs` != NULL selects the raw-scan form: scans_xy holds one float range per beam and the kernel forms the
// points itself (b2s_icp_batch_ranges), a quarter of the bytes of the float64 pair form.
struct IcpBufs {
    Buf &scans, &T, &iters, &cs;
};

static int icp_sequence_enqueue(b2s_icp *c, Trace &tr, const void *scans_xy, int is_f64, int scans, int n, int max_iter,
                                double tol, const double *beam_cs, double clamp, IcpBufs bufs, int force_chunks = 0)
{
    const size_t el = is_f64 ? 8 : 4, scan_bytes = (beam_cs ? (size_t)1 : (size_t)2) * n * el;
    const int pairs = scans - 1;
    int rc;
    if ((rc = bufs.scans.reserve((size_t)scans * scan_bytes))) return rc;
    if ((rc = bufs.T.reserve((size_t)pairs * 9 * sizeof(double)))) return rc;
    if ((rc = bufs.iters.reserve((size_t)pairs * sizeof(int32_t)))) return rc;
    if (beam_cs) {
        if ((rc = bufs.cs.reserve((size_t)n * 2 * sizeof(double)))) return rc;
        B2S_CUDA(cudaMemcpyAsync(bufs.cs.p, beam_cs, (size_t)n * 2 * sizeof(double), cudaMemcpyHostToDevice, c->copy_stream));
    }
    int want = (int)(((size_t)scans * scan_bytes + (8u << 20) - 1) / (8u << 20));  // ~8 MB of points per chunk
    if (beam_cs && want < 4 && pairs >= 4096) want = 4;  // (raw scans are half the bytes: keep the pipeline depth)
    if (force_chunks > 0) want = force_chunks;
    const int nchunk = pipeline_chunks(want, 8, pairs);
    char *d_scans = (char *)bufs.scans.p;
    // chunk k solves pairs [p0, p1) and therefore needs scans [p0, p1]; scan p0 arrived with the previous chunk
    auto upload = [&](int k, size_t p0, size_t p1, cudaStream_t st) -> int {
        const size_t s0 = k == 0 ? 0 : p0 + 1;
        B2S_CUDA(cudaMemcpyAsync(d_scans + s0 * scan_bytes, (const char *)scans_xy + s0 * scan_bytes, (p1 + 1 - s0) * scan_bytes,
                                 cudaMemcpyHostToDevice, st));
        return B2S_OK;
    };
    auto solve = [&](int, size_t p0, size_t p1, cudaStream_t ks) {
        const char *tar = d_scans + p0 * scan_bytes;
        double *dT = (double *)bufs.T.p + p0 * 9;
        int32_t *dI = (int32_t *)bufs.iters.p + p0;
        if (beam_cs)
            return b2s_icp_batch_ranges((const float *)tar, (const float *)(tar + scan_bytes), (const double *)bufs.cs.p, clamp,
                                        (int)(p1 - p0), n, max_iter, tol, dT, dI, ks);
        if (is_f64)
            return b2s_icp_batch_f64((const double *)tar, (const double *)(tar + scan_bytes), (int)(p1 - p0), n, n, max_iter, tol,
                                     dT, dI, ks);
        return b2s_icp_batch_f32((const float *)tar, (const float *)(tar + scan_bytes), (int)(p1 - p0), n, n, max_iter, tol,
                                 dT, dI, ks);
    };
    return icp_pipeline(c, tr, pairs, nchunk, upload, solve);
}

// Ending of the blocking sequence calls: optional pose chain and trajectory, then transforms and iteration counts.
static int icp_sequence_finish(b2s_icp *c, Trace &tr, int scans, const double *state, double *traj_out, double *T_out,
                               int32_t *iters_out)
{
    const int pairs = scans - 1;
    int rc;
    if (traj_out) {
        if ((rc = c->d_aux.reserve((size_t)scans * 3 * sizeof(double)))) return rc;
        if ((rc = b2s_pose_chain((const double *)c->d_T.p, pairs, state[0], state[1], state[2], (double *)c->d_aux.p, c->stream)))
            return rc;
        tr.mark("pose chain done", 0, c->stream);
        B2S_CUDA(cudaMemcpyAsync(traj_out, c->d_aux.p, (size_t)scans * 3 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    }
    return icp_read_back(c, tr, pairs, T_out, iters_out);
}

extern "C" int b2s_icp_process_sequence(b2s_icp *c, const void *scans_xy, int is_f64, int scans, int n,
                                        int max_iter, double tol, double *T_out, int32_t *iters_out)
{
    B2S_REQUIRE(c, "b2s_icp_process_sequence: null handle");
    B2S_REQUIRE(scans >= 0 && n > 0 && max_iter >= 0, "b2s_icp_process_sequence: bad sizes");
    if (scans <= 1) return B2S_OK;
    B2S_REQUIRE(scans_xy && T_out, "b2s_icp_process_sequence: null pointer");
    DeviceGuard g(c->device);
    Trace tr(c->stream);
    IcpBufs own = {c->d_tar, c->d_T, c->d_iters, c->d_src};
    int rc = icp_sequence_enqueue(c, tr, scans_xy, is_f64, scans, n, max_iter, tol, nullptr, 0.0, own);
    if (rc) return rc;
    return icp_sequence_finish(c, tr, scans, nullptr, nullptr, T_out, iters_out);
}

// The whole W9 LiDAR-odometry loop for a recorded stream: the K - 1 scan-to-scan transforms (above) and the pose
// chain xOdom (+)= T of [LOC9]:79-83 / [ICP]:185-190 as a parallel prefix over them, without the transforms leaving
// the device in between.  traj_out [scans][3] starts at (x0, y0, th0); T_out / iters_out may be NULL.
extern "C" int b2s_icp_odometry(b2s_icp *c, const void *scans_xy, int is_f64, int scans, int n, int max_iter,
                                double tol, double x0, double y0, double th0, double *traj_out, double *T_out,
                                int32_t *iters_out)
{
    B2S_REQUIRE(c, "b2s_icp_odometry: null handle");
    B2S_REQUIRE(scans >= 1 && n > 0 && max_iter >= 0, "b2s_icp_odometry: bad sizes");
    B2S_REQUIRE(traj_out && (scans_xy || scans == 1), "b2s_icp_odometry: null pointer");
    DeviceGuard g(c->device);
    Trace tr(c->stream);
    int rc;
    IcpBufs own = {c->d_tar, c->d_T, c->d_iters, c->d_src};
    if (scans > 1 && (rc = icp_sequence_enqueue(c, tr, scans_xy, is_f64, scans, n, max_iter, tol, nullptr, 0.0, own))) return rc;
    const double state[3] = {x0, y0, th0};
    return icp_sequence_finish(c, tr, scans, state, traj_out, T_out, iters_out);
}

// The same loop fed with what the sensor delivers: ranges [scans][n] (sensor_msgs/LaserScan.ranges) and the beam
// table [n][2] = cos, sin of linspace(angle_min, angle_max, n).  laserToNumpy ([ICP]:216-229; with clamp_inf_to > 0
// the W12 form [SLAM]:115-123) runs inside the ICP kernel in float64, so 4 bytes per beam cross PCIe instead of the 8
// (float32 points) or 16 (the reference's float64 points).  state / traj_out may both be NULL (no pose chain).
extern "C" int b2s_icp_process_scans(b2s_icp *c, const float *ranges, const double *beam_cs, double clamp_inf_to,
                                     int scans, int n, int max_iter, double tol, const double *state3,
                                     double *traj_out, double *T_out, int32_t *iters_out)
{
    B2S_REQUIRE(c, "b2s_icp_process_scans: null handle");
    B2S_REQUIRE(scans >= 0 && n > 0 && max_iter >= 0, "b2s_icp_process_scans: bad sizes");
    B2S_REQUIRE((traj_out == nullptr) == (state3 == nullptr), "b2s_icp_process_scans: state and traj_out go together");
    if (scans == 0 || (scans == 1 && !traj_out)) return B2S_OK;
    B2S_REQUIRE(ranges && beam_cs && (T_out || traj_out), "b2s_icp_process_scans: null pointer");
    B2S_REQUIRE(clamp_inf_to == clamp_inf_to, "b2s_icp_process_scans: NaN clamp");
    DeviceGuard g(c->device);
    Trace tr(c->stream);
    int rc;
    IcpBufs own = {c->d_tar, c->d_T, c->d_iters, c->d_src};
    if (scans > 1 && (rc = icp_sequence_enqueue(c, tr, ranges, 0, scans, n, max_iter, tol, beam_cs, clamp_inf_to, own))) return rc;
    return icp_sequence_finish(c, tr, scans, state3, traj_out, T_out, iters_out);
}

// Streaming forms of b2s_icp_process_sequence / b2s_icp_process_scans: submit enqueues the uploads and the solves of a
// scan stream on the slot's own device buffers and the read-back of its transforms on a third stream, and returns a
// ticket; two calls may be in flight, so the scans of call k + 1 cross PCIe while call k is being solved.
static int icp_submit(b2s_icp *c, const void *scans_data, int is_f64, const double *beam_cs, double clamp, int scans, int n,
                      int max_iter, double tol, double *T_out, int32_t *iters_out, int *ticket_out)
{
    DeviceGuard g(c->device);
    const int ticket = c->submitted;
    IcpSlot &sl = c->slot[ticket & 1];
    IcpSlot &other = c->slot[(ticket & 1) ^ 1];
    if (sl.in_flight) {
        B2S_CUDA(cudaEventSynchronize(sl.done));
        sl.in_flight = false;
    }
    const int pairs = scans - 1;
    Trace tr(c->stream);
    B2S_CUDA(cudaStreamWaitEvent(c->copy_stream, sl.inputs_free, 0));
    IcpBufs bufs = {sl.d_scans, sl.d_T, sl.d_iters, sl.d_cs};
    int rc;
    // while the other slot is being solved this call's upload is hidden anyway: fewer, larger chunks
    if (pairs > 0 && (rc = icp_sequence_enqueue(c, tr, scans_data, is_f64, scans, n, max_iter, tol, beam_cs, clamp, bufs,
                                                other.in_flight ? 2 : 0)))
        return rc;
    B2S_CUDA(cudaEventRecord(sl.inputs_free, c->stream));
    B2S_CUDA(cudaEventRecord(c->handoff, c->stream));
    B2S_CUDA(cudaStreamWaitEvent(c->d2h_stream, c->handoff, 0));
    if (pairs > 0) {
        B2S_CUDA(cudaMemcpyAsync(T_out, sl.d_T.p, (size_t)pairs * 9 * sizeof(double), cudaMemcpyDeviceToHost, c->d2h_stream));
        if (iters_out)
            B2S_CUDA(cudaMemcpyAsync(iters_out, sl.d_iters.p, (size_t)pairs * sizeof(int32_t), cudaMemcpyDeviceToHost, c->d2h_stream));
    }
    B2S_CUDA(cudaEventRecord(sl.done, c->d2h_stream));
    sl.in_flight = true;
    sl.ticket = ticket;
    c->submitted = ticket + 1;
    *ticket_out = ticket;
    return B2S_OK;
}

extern "C" int b2s_icp_submit_sequence(b2s_icp *c, const void *scans_xy, int is_f64, int scans, int n, int max_iter,
                                       double tol, double *T_out, int32_t *iters_out, int *ticket_out)
{
    B2S_REQUIRE(c && ticket_out, "b2s_icp_submit_sequence: null pointer");
    B2S_REQUIRE(scans >= 0 && n > 0 && max_iter >= 0, "b2s_icp_submit_sequence: bad sizes");
    B2S_REQUIRE(scans <= 1 || (scans_xy && T_out), "b2s_icp_submit_sequence: null pointer");
    return icp_submit(c, scans_xy, is_f64, nullptr, 0.0, scans < 1 ? 1 : scans, n, max_iter, tol, T_out, iters_out, ticket_out);
}

extern "C" int b2s_icp_submit_scans(b2s_icp *c, const float *ranges, const double *beam_cs, double clamp_inf_to, int scans,
                                    int n, int max_iter, double tol, double *T_out, int32_t *iters_out, int *ticket_out)
{
    B2S_REQUIRE(c && ticket_out, "b2s_icp_submit_scans: null pointer");
    B2S_REQUIRE(scans >= 0 && n > 0 && max_iter >= 0, "b2s_icp_submit_scans: bad sizes");
    B2S_REQUIRE(scans <= 1 || (ranges && beam_cs && T_out), "b2s_icp_submit_scans: null pointer");
    B2S_REQUIRE(clamp_inf_to == clamp_inf_to, "b2s_icp_submit_scans: NaN clamp");
    return icp_submit(c, ranges, 0, beam_cs, clamp_inf_to, scans < 1 ? 1 : scans, n, max_iter, tol, T_out, iters_out, ticket_out);
}

extern "C" int b2s_icp_wait(b2s_icp *c, int ticket)
{
    B2S_REQUIRE(c, "b2s_icp_wait: null handle");
    B2S_REQUIRE(ticket >= 0 && ticket < c->submitted, "b2s_icp_wait: unknown ticket");
    DeviceGuard g(c->device);
    IcpSlot &sl = c->slot[ticket & 1];
    if (!sl.in_flight || sl.ticket != ticket) return B2S_OK;
    B2S_CUDA(cudaEventSynchronize(sl.done));
    sl.in_flight = false;
    return B2S_OK;
}

static const char NAN_TO_INT[] = "cannot convert float NaN to integer";  // int(nan) in the reference

extern "C" int b2s_icp_set_map(b2s_icp *c, const double *obs_x, const double *obs_y, int count)
{
    B2S_REQUIRE(c, "b2s_icp_set_map: null handle");
    B2S_REQUIRE(count >= 0 && (count == 0 || (obs_x && obs_y)), "b2s_icp_set_map: bad arguments");
    c->map_count = 0;
    for (int i = 0; i < count; ++i)
        if (obs_x[i] != obs_x[i] || obs_y[i] != obs_y[i]) {
            set_error("%s", NAN_TO_INT);
            return B2S_ERR_NONFINITE;
        }
    if (count == 0) return B2S_OK;
    DeviceGuard g(c->device);
    int rc;
    if ((rc = c->d_map.reserve((size_t)count * 2 * sizeof(double)))) return rc;
    double *d = (double *)c->d_map.p;
    B2S_CUDA(cudaMemcpyAsync(d, obs_x, (size_t)count * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    B2S_CUDA(cudaMemcpyAsync(d + count, obs_y, (size_t)count * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    B2S_CUDA(cudaStreamSynchronize(c->stream));
    c->map_count = count;
    return B2S_OK;
}

// The ranges and poses go through icp_pipeline.  Per chunk: the virtual scans straight into the target layout,
// laserToNumpy of the ranges into the source layout, then the float64 ICP on the two.
extern "C" int b2s_icp_map_observation(b2s_icp *c, const float *ranges, const double *poses3, const double *beam_cs,
                                       double clamp_inf_to, int scans, int n, double angle_min, double angle_increment,
                                       double far_range, int max_iter, double tol, double *T_out, int32_t *iters_out,
                                       double *virtual_out)
{
    B2S_REQUIRE(c, "b2s_icp_map_observation: null handle");
    B2S_REQUIRE(scans >= 0 && n > 0 && max_iter >= 0, "b2s_icp_map_observation: bad sizes");
    B2S_REQUIRE(n <= ICP_MAX_POINTS, "b2s_icp_batch: more than 2304 source points per scan is not supported");
    B2S_REQUIRE(c->map_count > 0, "b2s_icp_map_observation: no static map set (b2s_icp_set_map)");
    if (scans == 0) return B2S_OK;
    B2S_REQUIRE(ranges && poses3 && beam_cs && T_out, "b2s_icp_map_observation: null pointer");
    B2S_REQUIRE(clamp_inf_to == clamp_inf_to && tol == tol, "b2s_icp_map_observation: NaN clamp / tolerance");
    B2S_REQUIRE(angle_increment != 0.0 && angle_increment == angle_increment, "b2s_icp_map_observation: angle_increment");
    // the reference's int() raises on the first obstacle's bin of a NaN pose; +-inf poses only give bins no obstacle wins
    for (size_t i = 0; i < (size_t)scans * 3; ++i)
        if (poses3[i] != poses3[i]) {
            set_error("%s", NAN_TO_INT);
            return B2S_ERR_NONFINITE;
        }
    DeviceGuard g(c->device);
    Trace tr(c->stream);
    const size_t cs_bytes = (size_t)n * 2 * sizeof(double), pose_bytes = (size_t)scans * 3 * sizeof(double);
    const size_t pose_off = cs_bytes, range_off = (pose_off + pose_bytes + 15) & ~(size_t)15;
    const size_t cloud = (size_t)scans * 2 * n;  // doubles of one cloud set
    int rc;
    if ((rc = c->d_map_in.reserve(range_off + (size_t)scans * n * sizeof(float)))) return rc;
    if ((rc = c->d_map_tar.reserve((cloud + (virtual_out ? (size_t)scans * n : 0)) * sizeof(double)))) return rc;
    if ((rc = c->d_map_src.reserve(cloud * sizeof(double)))) return rc;
    if ((rc = c->d_T.reserve((size_t)scans * 9 * sizeof(double)))) return rc;
    if ((rc = c->d_iters.reserve((size_t)scans * sizeof(int32_t)))) return rc;
    char *in = (char *)c->d_map_in.p;
    const double *d_cs = (const double *)in, *d_pose = (const double *)(in + pose_off);
    const float *d_ranges = (const float *)(in + range_off);
    double *d_tar = (double *)c->d_map_tar.p, *d_src = (double *)c->d_map_src.p, *d_virt = virtual_out ? d_tar + cloud : nullptr;
    const double *map_x = (const double *)c->d_map.p, *map_y = map_x + c->map_count;
    // at most ~8 MB of uploads and ~2500 scans per chunk (about three waves of ICP CTAs).  Measured on the course map,
    // 360 beams (profiles/r6): 3000 scans 0.932 / 0.906 / 0.966 ms at 1 / 2 / 4 chunks, 9999 scans 2.79 / 2.69 / 2.63 ms
    // at 1 / 2 / 4 chunks
    int want = (int)(((size_t)scans * ((size_t)n * sizeof(float) + 3 * sizeof(double)) + (8u << 20) - 1) / (8u << 20));
    if (want < (scans + 2499) / 2500) want = (scans + 2499) / 2500;
    const int nchunk = pipeline_chunks(want, 8, scans);
    B2S_CUDA(cudaMemcpyAsync(in, beam_cs, cs_bytes, cudaMemcpyHostToDevice, c->copy_stream));
    auto upload = [&](int, size_t s0, size_t s1, cudaStream_t st) -> int {
        B2S_CUDA(cudaMemcpyAsync(in + pose_off + s0 * 3 * sizeof(double), poses3 + s0 * 3, (s1 - s0) * 3 * sizeof(double),
                                 cudaMemcpyHostToDevice, st));
        B2S_CUDA(cudaMemcpyAsync(in + range_off + s0 * n * sizeof(float), ranges + s0 * n, (s1 - s0) * n * sizeof(float),
                                 cudaMemcpyHostToDevice, st));
        return B2S_OK;
    };
    auto solve = [&](int k, size_t s0, size_t s1, cudaStream_t ks) {
        const int ns = (int)(s1 - s0);
        double *tar = d_tar + s0 * 2 * n, *src = d_src + s0 * 2 * n;
        if ((rc = b2s_virtual_scan_batch(map_x, map_y, c->map_count, d_pose + s0 * 3, ns, angle_min, angle_increment, n,
                                         far_range, d_cs, d_virt ? d_virt + s0 * n : nullptr, tar, ks)))
            return rc;
        tr.mark("virtual scan chunk done", k, ks);
        if ((rc = laser_points(d_ranges + s0 * n, d_cs, clamp_inf_to, ns, n, src, ks))) return rc;
        return b2s_icp_batch_f64(tar, src, ns, n, n, max_iter, tol, (double *)c->d_T.p + s0 * 9,
                                 (int32_t *)c->d_iters.p + s0, ks);
    };
    if ((rc = icp_pipeline(c, tr, scans, nchunk, upload, solve))) return rc;
    if (virtual_out)
        B2S_CUDA(cudaMemcpyAsync(virtual_out, d_virt, (size_t)scans * n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    return icp_read_back(c, tr, scans, T_out, iters_out);
}

// Relocalization: the map observation of every scan at every candidate.  The H virtual scans depend on the candidate
// only, so they are built once into the target layout and shared by all scans; per scan, laserToNumpy forms its source
// cloud once, replicated into the H source rows, and the H-pair ICP runs with its score output, the scans alternating
// between stream and stream2.  One selection launch over all scans follows on stream, then the read-back.
extern "C" int b2s_icp_relocalize(b2s_icp *c, const float *ranges, const double *candidates3, const double *beam_cs,
                                  double clamp_inf_to, int scans, int hyps, int n, double angle_min, double angle_increment,
                                  double far_range, int max_iter, double tol, int32_t *best_out, double *pose_out,
                                  double *score_out, int32_t *iters_out, double *T_out)
{
    B2S_REQUIRE(scans >= 0 && hyps > 0 && n > 0 && max_iter >= 0 && (long long)scans * hyps <= 0x7fffffffLL,
                "b2s_icp_relocalize: bad sizes");
    B2S_REQUIRE(n <= ICP_MAX_POINTS, "b2s_icp_batch: more than 2304 source points per scan is not supported");
    B2S_REQUIRE(angle_increment != 0.0 && angle_increment == angle_increment, "b2s_icp_relocalize: angle_increment");
    B2S_REQUIRE(clamp_inf_to == clamp_inf_to && tol == tol, "b2s_icp_relocalize: NaN clamp / tolerance");
    B2S_REQUIRE(c, "b2s_icp_relocalize: null handle");
    B2S_REQUIRE(c->map_count > 0, "b2s_icp_relocalize: no static map set (b2s_icp_set_map)");
    if (scans == 0) return B2S_OK;
    B2S_REQUIRE(ranges && candidates3 && beam_cs && best_out && pose_out, "b2s_icp_relocalize: null pointer");
    for (size_t i = 0; i < (size_t)hyps * 3; ++i)  // as in b2s_icp_map_observation
        if (candidates3[i] != candidates3[i]) {
            set_error("%s", NAN_TO_INT);
            return B2S_ERR_NONFINITE;
        }
    DeviceGuard g(c->device);
    Trace tr(c->stream);
    const size_t H = (size_t)hyps, K = (size_t)scans, cloud = H * 2 * n;  // doubles of one set of H clouds
    const size_t cs_bytes = (size_t)n * 2 * sizeof(double), cand_bytes = H * 3 * sizeof(double);
    const size_t cand_off = cs_bytes, range_off = (cand_off + cand_bytes + 15) & ~(size_t)15;
    // d_aux: scores [K][H] | best [K] | poses [K][3] (+ one scan's source cloud per compute stream)
    const size_t score_bytes = K * H * sizeof(double), best_off = score_bytes;
    const size_t pose_off = (best_off + K * sizeof(int32_t) + 15) & ~(size_t)15, cloud_off = pose_off + K * 3 * sizeof(double);
    int rc;
    if ((rc = c->d_map_in.reserve(range_off + K * n * sizeof(float)))) return rc;
    if ((rc = c->d_map_tar.reserve(cloud * sizeof(double)))) return rc;
    if ((rc = c->d_map_src.reserve(2 * cloud * sizeof(double)))) return rc;
    if ((rc = c->d_T.reserve(K * H * 9 * sizeof(double)))) return rc;
    if ((rc = c->d_iters.reserve(K * H * sizeof(int32_t)))) return rc;
    if ((rc = c->d_aux.reserve(cloud_off + 2 * cs_bytes))) return rc;
    char *in = (char *)c->d_map_in.p, *aux = (char *)c->d_aux.p;
    const double *d_cs = (const double *)in, *d_cand = (const double *)(in + cand_off);
    const float *d_ranges = (const float *)(in + range_off);
    double *d_tar = (double *)c->d_map_tar.p, *d_T = (double *)c->d_T.p, *d_score = (double *)aux;
    int32_t *d_iters = (int32_t *)c->d_iters.p, *d_best = (int32_t *)(aux + best_off);
    double *d_pose = (double *)(aux + pose_off);
    const double *map_x = (const double *)c->d_map.p, *map_y = map_x + c->map_count;
    // (every call ends with a synchronize, so the device buffers are free to overwrite here)
    B2S_CUDA(cudaMemcpyAsync(in, beam_cs, cs_bytes, cudaMemcpyHostToDevice, c->stream));
    B2S_CUDA(cudaMemcpyAsync(in + cand_off, candidates3, cand_bytes, cudaMemcpyHostToDevice, c->stream));
    B2S_CUDA(cudaMemcpyAsync(in + range_off, ranges, K * n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    if ((rc = b2s_virtual_scan_batch(map_x, map_y, c->map_count, d_cand, hyps, angle_min, angle_increment, n, far_range,
                                     d_cs, nullptr, d_tar, c->stream)))
        return rc;
    tr.mark("virtual scans done", 0, c->stream);
    B2S_CUDA(cudaEventRecord(c->chunk_ready[0], c->stream));  // the uploads and targets, for stream2
    B2S_CUDA(cudaStreamWaitEvent(c->stream2, c->chunk_ready[0], 0));
    for (size_t k = 0; k < K; ++k) {
        cudaStream_t ks = (k & 1) ? c->stream2 : c->stream;
        double *one = (double *)(aux + cloud_off) + (k & 1) * 2 * n, *src = (double *)c->d_map_src.p + (k & 1) * cloud;
        if ((rc = laser_points(d_ranges + k * n, d_cs, clamp_inf_to, 1, n, one, ks))) return rc;
        if ((rc = replicate_row(one, (size_t)2 * n, H, src, ks))) return rc;
        if ((rc = b2s_icp_batch_f64_err(d_tar, src, hyps, n, n, max_iter, tol, d_T + k * H * 9, d_iters + k * H,
                                        d_score + k * H, ks)))
            return rc;
        tr.mark("relocalize scan done", (int)k, ks);
    }
    if (K > 1) {
        B2S_CUDA(cudaEventRecord(c->joined, c->stream2));
        B2S_CUDA(cudaStreamWaitEvent(c->stream, c->joined, 0));
    }
    if ((rc = b2s_relocalize_select(d_score, d_T, d_cand, scans, hyps, d_best, d_pose, c->stream))) return rc;
    tr.mark("select done", 0, c->stream);
    B2S_CUDA(cudaMemcpyAsync(best_out, d_best, K * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    B2S_CUDA(cudaMemcpyAsync(pose_out, d_pose, K * 3 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (score_out) B2S_CUDA(cudaMemcpyAsync(score_out, d_score, score_bytes, cudaMemcpyDeviceToHost, c->stream));
    return icp_read_back(c, tr, (int)(K * H), T_out, iters_out);
}

extern "C" int b2s_icp_find_nearest(b2s_icp *c, const double *src_xy, int n, const double *tar_xy,
                                    int m, double *dist_out, int64_t *idx_out)
{
    B2S_REQUIRE(c, "b2s_icp_find_nearest: null handle");
    B2S_REQUIRE(n >= 0 && m >= 0, "b2s_icp_find_nearest: negative size");
    if (n == 0) return B2S_OK;
    B2S_REQUIRE(src_xy && dist_out && idx_out && (tar_xy || m == 0), "b2s_icp_find_nearest: null pointer");
    DeviceGuard g(c->device);
    int rc;
    if ((rc = c->d_src.reserve((size_t)n * 16))) return rc;
    if ((rc = c->d_tar.reserve((size_t)(m > 0 ? m : 1) * 16))) return rc;
    if ((rc = c->d_T.reserve((size_t)n * 8))) return rc;
    if ((rc = c->d_aux.reserve((size_t)n * 8))) return rc;
    B2S_CUDA(cudaMemcpyAsync(c->d_src.p, src_xy, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
    if (m > 0) B2S_CUDA(cudaMemcpyAsync(c->d_tar.p, tar_xy, (size_t)m * 16, cudaMemcpyHostToDevice, c->stream));
    rc = b2s_nearest_f64((const double *)c->d_src.p, n, (const double *)c->d_tar.p, m, (double *)c->d_T.p,
                         (int64_t *)c->d_aux.p, c->stream);
    if (rc) return rc;
    B2S_CUDA(cudaMemcpyAsync(dist_out, c->d_T.p, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
    B2S_CUDA(cudaMemcpyAsync(idx_out, c->d_aux.p, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
    B2S_CUDA(cudaStreamSynchronize(c->stream));
    return B2S_OK;
}

extern "C" int b2s_icp_get_transform(b2s_icp *c, const double *src_xy, const double *tar_xy, int n,
                                     double *T_out)
{
    B2S_REQUIRE(c, "b2s_icp_get_transform: null handle");
    B2S_REQUIRE(n > 0 && src_xy && tar_xy && T_out, "b2s_icp_get_transform: bad arguments");
    DeviceGuard g(c->device);
    int rc;
    if ((rc = c->d_src.reserve((size_t)n * 16))) return rc;
    if ((rc = c->d_tar.reserve((size_t)n * 16))) return rc;
    if ((rc = c->d_T.reserve(9 * 8))) return rc;
    B2S_CUDA(cudaMemcpyAsync(c->d_src.p, src_xy, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
    B2S_CUDA(cudaMemcpyAsync(c->d_tar.p, tar_xy, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream));
    rc = b2s_rigid_fit_f64((const double *)c->d_src.p, (const double *)c->d_tar.p, n, (double *)c->d_T.p, c->stream);
    if (rc) return rc;
    B2S_CUDA(cudaMemcpyAsync(T_out, c->d_T.p, 9 * 8, cudaMemcpyDeviceToHost, c->stream));
    B2S_CUDA(cudaStreamSynchronize(c->stream));
    return B2S_OK;
}

// ------------------------------------------------------------------------------ Mapping object

extern "C" int b2s_mapping_create(b2s_mapping **out, int xw, int yw, double xyreso, double w_hit,
                                  double w_miss, double thresh, int device)
{
    B2S_REQUIRE(out, "b2s_mapping_create: null pointer");
    *out = nullptr;
    B2S_REQUIRE(xw > 0 && yw > 0 && (long long)xw * yw < (1ll << 30), "b2s_mapping_create: grid size");
    B2S_REQUIRE(xyreso > 0.0 && isfinite(xyreso), "b2s_mapping_create: xyreso must be positive");
    int ndev = 0;
    B2S_CUDA(cudaGetDeviceCount(&ndev));
    if (ndev <= 0) {
        set_error("no CUDA device");
        return B2S_ERR_CUDA;
    }
    if (device < 0) B2S_CUDA(cudaGetDevice(&device));
    B2S_REQUIRE(device < ndev, "b2s_mapping_create: device index out of range");
    DeviceGuard g(device);
    b2s_mapping *m = new (std::nothrow) b2s_mapping();
    if (!m) return B2S_ERR_NOMEM;
    m->device = device;
    m->xw = xw;
    m->yw = yw;
    m->xyreso = xyreso;
    // generalisation of the literals of [MAP]:33-36; exactly 10.0 / 10.0 at (200, 200, 0.1)
    m->cells_per_m = 1.0 / xyreso;
    m->off_x = (double)xw * xyreso / 2.0;
    m->off_y = (double)yw * xyreso / 2.0;
    m->w_hit = w_hit;
    m->w_miss = w_miss;
    m->thresh = thresh;
    const size_t plane = (size_t)xw * yw * sizeof(int32_t);
    cudaError_t e = m->create();
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->begun, cudaEventDisableTiming);
    for (MappingSlot &sl : m->slot) {
        if (e == cudaSuccess) e = cudaMalloc((void **)&sl.d_cnt, B2S_CNT_WORDS * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMallocHost((void **)&sl.h_cnt, B2S_CNT_WORDS * sizeof(int32_t));
    }
    if (e == cudaSuccess) e = cudaMalloc((void **)&m->hit, plane);
    if (e == cudaSuccess) e = cudaMalloc((void **)&m->miss, plane);
    if (e == cudaSuccess) e = cudaMalloc((void **)&m->counters, 2 * B2S_CNT_WORDS * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMalloc(&m->workspace, b2s_grid_workspace_bytes(xw, yw));
    if (e == cudaSuccess && b2s_grid_workspace_init(m->workspace, xw, yw, m->stream) != B2S_OK) e = cudaErrorUnknown;
    if (e == cudaSuccess) e = cudaMemsetAsync(m->hit, 0, plane, m->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->miss, 0, plane, m->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(m->counters, 0, 2 * B2S_CNT_WORDS * sizeof(int32_t), m->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(m->stream);
    if (e != cudaSuccess) {
        int rc = cuda_fail(e, "b2s_mapping_create");
        b2s_mapping_destroy(m);
        return e == cudaErrorMemoryAllocation ? B2S_ERR_NOMEM : rc;
    }
    *out = m;
    return B2S_OK;
}

extern "C" int b2s_mapping_destroy(b2s_mapping *m)
{
    if (!m) return B2S_OK;
    DeviceGuard g(m->device);
    m->teardown([m] {
        if (m->hit) cudaFree(m->hit);
        if (m->miss) cudaFree(m->miss);
        if (m->counters) cudaFree(m->counters);
        if (m->workspace) cudaFree(m->workspace);
        if (m->h_packed) cudaFreeHost(m->h_packed);
        if (m->h_ids) cudaFreeHost(m->h_ids);
        m->d_packed.release();
        m->d_in.release(); m->d_datamap.release(); m->d_pmap.release();
        m->h_pose.release();
        for (MappingSlot &sl : m->slot) {
            sl.d_in.release(); sl.d_map.release(); sl.h_pose.release();
            if (sl.d_cnt) cudaFree(sl.d_cnt);
            if (sl.h_cnt) cudaFreeHost(sl.h_cnt);
        }
        if (m->begun) cudaEventDestroy(m->begun);
    });
    delete m;
    return B2S_OK;
}

extern "C" int b2s_mapping_reset(b2s_mapping *m)
{
    B2S_REQUIRE(m, "b2s_mapping_reset: null handle");
    DeviceGuard g(m->device);
    const size_t plane = (size_t)m->xw * m->yw * sizeof(int32_t);
    B2S_CUDA(cudaMemsetAsync(m->hit, 0, plane, m->stream));
    B2S_CUDA(cudaMemsetAsync(m->miss, 0, plane, m->stream));
    B2S_CUDA(cudaStreamSynchronize(m->stream));
    m->pmap_valid = false;
    return B2S_OK;
}

namespace {
// The verdict on a batch from its ray-cast's B2S_CNT_* words: a coordinate the reference's int() raises on, or a beam
// too long to march, rejects the whole batch.
bool batch_rejected(const int32_t *cnt)
{
    return cnt[B2S_CNT_NONFINITE] || cnt[B2S_CNT_OVERFLOW] || cnt[B2S_CNT_TOO_LONG] > 0;
}

// Status and message of a rejected batch.  The reference raises at the first offending beam in scan order; NaN and
// inf map to different exception classes, NaN wins when both occur (documented deviation).
int batch_error(const int32_t *cnt)
{
    if (cnt[B2S_CNT_NONFINITE] || cnt[B2S_CNT_OVERFLOW]) {
        set_error(cnt[B2S_CNT_NONFINITE] ? "cannot convert float NaN to integer" : "cannot convert float infinity to integer");
        return B2S_ERR_NONFINITE;
    }
    set_error("%d beam(s) longer than %d cells: batch rejected", cnt[B2S_CNT_TOO_LONG], B2S_MAX_PATH_CELLS);
    return B2S_ERR_TOO_LONG;
}

// Mapping.update for a batch, all-or-nothing like a Python exception raised before the loop.
//   * the batch is cut into up to 16 chunks of scans; chunk k+1 crosses PCIe on the copy stream while
//     chunk k is screened and ray-cast on the compute stream
//   * beams that int() would raise on ([MAP]:33-36) are skipped and counted by the kernels, so applying
//     a chunk before the verdict on the whole batch is known is safe: a rejected batch is taken back
//     out with the sign -1 kernel (integer adds: exact inverse)
constexpr int PACK_CAP = 1024;  // dirty tiles shipped individually; beyond that the whole map is cheaper

int mapping_update_impl(b2s_mapping *m, const HostBatch &hb, int scans, int beams, int8_t *pmap_out,
                        bool incremental = false, int32_t *tiles_out = nullptr, int tiles_cap = 0,
                        int *tiles_count = nullptr)
{
    DeviceGuard g(m->device);
    for (int k = 0; k < 2; ++k)  // streamed steps still in flight land first (their verdicts belong to their tickets)
        if (m->slot[k].in_flight) B2S_CUDA(cudaEventSynchronize(m->slot[k].done));
    Trace tr(m->stream);
    const size_t total = (size_t)scans * beams;
    int rc;
    DeviceBatch db(hb, scans, beams);
    if (total > 0) {
        if ((rc = m->d_in.reserve(db.bytes()))) return rc;
        db.bind(m->d_in.p);
        // counters[0..3]: the ray-cast kernel's own (B2S_CNT_*); counters[4]: dirty-tile count of this call
        B2S_CUDA(cudaMemsetAsync(m->counters, 0, 2 * B2S_CNT_WORDS * sizeof(int32_t), m->stream));
        // the dirty-tile map describes THIS call
        B2S_CUDA(cudaMemsetAsync((char *)m->workspace + GRID_WS_HEADER, 0, grid_dirty_bytes(m->xw, m->yw), m->stream));
        // ~1M beams per chunk: with consecutive chunks overlapping on two compute streams an extra launch costs
        // little, and the first ray-cast starts after 1/16 of the copy (measured: profiles/scripts/chunk_sweep.py)
        const int nchunk = pipeline_chunks((int)((total * (db.el() / sizeof(float)) + (1u << 20) - 1) >> 20), MAX_CHUNKS, scans);
        if (nchunk > 1) {  // the second compute stream starts after the resets above (single-chunk calls never use it)
            B2S_CUDA(cudaEventRecord(m->begun, m->stream));
            B2S_CUDA(cudaStreamWaitEvent(m->stream2, m->begun, 0));
        }
        if (hb.fused && hb.poses3 && (rc = m->h_pose.reserve((size_t)scans * 4 * sizeof(double)))) return rc;
        // per chunk: copies on the copy stream -> ray-cast on a compute stream once they landed
        for (int k = 0; k < nchunk; ++k) {
            const size_t s0 = (size_t)scans * k / nchunk, s1 = (size_t)scans * (k + 1) / nchunk;
            cudaStream_t cs = m->copy_stream;
            if ((rc = db.upload(hb, s0, s1, (double *)m->h_pose.p, cs))) return rc;
            B2S_CUDA(cudaEventRecord(m->chunk_ready[k], cs));
            tr.mark("h2d chunk done", k, cs);
            // odd chunks run on the second compute stream; the last chunk (which also folds the scratch plane)
            // runs on the main stream after the second one has drained
            const bool last = (k == nchunk - 1);
            cudaStream_t ks = (!last && (k & 1)) ? m->stream2 : m->stream;
            if (last && nchunk > 1) {
                B2S_CUDA(cudaEventRecord(m->joined, m->stream2));
                B2S_CUDA(cudaStreamWaitEvent(m->stream, m->joined, 0));
            }
            B2S_CUDA(cudaStreamWaitEvent(ks, m->chunk_ready[k], 0));
            if ((rc = db.raycast(m, s0, s1, +1, m->counters, ks, last))) return rc;
            tr.mark("ray-cast chunk done", k, ks);
        }
    }
    int32_t cnt[2 * B2S_CNT_WORDS] = {0, 0, 0, 0, 0, 0, 0, 0};
    const size_t cells = (size_t)m->xw * m->yw;
    const size_t tile_bytes = (size_t)GRID_TILE * GRID_TILE;
    // Incremental read-back: when the host already holds the previous map and this call touched few tiles,
    // finalize and ship only those tiles (a single scan dirties ~20 of the 4096 tiles of a 4096^2 map).
    bool patched = false, have_cnt = false;
    if (tiles_count) *tiles_count = -1;
    if (pmap_out && incremental && m->pmap_valid && total > 0) {
        if ((rc = m->d_pmap.reserve(cells))) return rc;
        if ((rc = m->d_packed.reserve(PACK_CAP * tile_bytes + PACK_CAP * sizeof(int32_t)))) return rc;
        if (!m->h_packed) {
            B2S_CUDA(cudaMallocHost((void **)&m->h_packed, PACK_CAP * tile_bytes));
            B2S_CUDA(cudaMallocHost((void **)&m->h_ids, PACK_CAP * sizeof(int32_t)));
        }
        int8_t *d_packed = (int8_t *)m->d_packed.p;
        int32_t *d_ids = (int32_t *)((char *)m->d_packed.p + PACK_CAP * tile_bytes);
        rc = grid_finalize_dirty(m->hit, m->miss, m->xw, m->yw, m->w_hit, m->w_miss, m->thresh, m->workspace,
                                 (int8_t *)m->d_pmap.p, d_packed, d_ids, m->counters + B2S_CNT_WORDS, PACK_CAP, m->stream);
        if (rc) return rc;
        B2S_CUDA(cudaMemcpyAsync(cnt, m->counters, sizeof(cnt), cudaMemcpyDeviceToHost, m->stream));
        B2S_CUDA(cudaStreamSynchronize(m->stream));
        have_cnt = true;
        const int nd = cnt[B2S_CNT_WORDS];
        const bool bad = batch_rejected(cnt);
        if (!bad && nd <= PACK_CAP) {
            if (nd > 0) {
                B2S_CUDA(cudaMemcpyAsync(m->h_packed, d_packed, (size_t)nd * tile_bytes, cudaMemcpyDeviceToHost, m->stream));
                B2S_CUDA(cudaMemcpyAsync(m->h_ids, d_ids, (size_t)nd * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
                B2S_CUDA(cudaStreamSynchronize(m->stream));
            }
            const int tiles_y = grid_tiles(m->yw);
            for (int k = 0; k < nd; ++k) {
                const int tile = m->h_ids[k];
                const int x0 = (tile / tiles_y) * GRID_TILE, y0 = (tile % tiles_y) * GRID_TILE;
                const int nx = (m->xw - x0 < GRID_TILE) ? m->xw - x0 : GRID_TILE;
                const int ny = (m->yw - y0 < GRID_TILE) ? m->yw - y0 : GRID_TILE;
                for (int r = 0; r < nx; ++r)
                    memcpy(pmap_out + (size_t)(x0 + r) * m->yw + y0, m->h_packed + (size_t)k * tile_bytes + (size_t)r * GRID_TILE,
                           (size_t)ny);
                if (tiles_out && k < tiles_cap) tiles_out[k] = tile;
            }
            if (tiles_count) *tiles_count = (tiles_out && nd > tiles_cap) ? -1 : nd;
            patched = true;
        }
        if (bad) m->pmap_valid = false;  // handled (and rolled back) below with a full refresh
    }
    const bool cnt_pending = !have_cnt && total > 0;
    if (pmap_out && !patched) {
        if ((rc = m->d_pmap.reserve(cells))) return rc;
        rc = b2s_grid_finalize(m->hit, m->miss, m->xw, m->yw, m->w_hit, m->w_miss, m->thresh, nullptr,
                               (int8_t *)m->d_pmap.p, m->stream);
        if (rc) return rc;
        tr.mark("finalize done", 0, m->stream);
        B2S_CUDA(cudaMemcpyAsync(pmap_out, m->d_pmap.p, cells, cudaMemcpyDeviceToHost, m->stream));
        tr.mark("map d2h done", 0, m->stream);
        m->pmap_valid = true;
    } else if (!pmap_out) {
        m->pmap_valid = false;  // counts moved on without the device map
    }
    // (a pageable destination makes this copy synchronous, so it goes last: everything else is already queued)
    if (cnt_pending) B2S_CUDA(cudaMemcpyAsync(cnt, m->counters, sizeof(cnt), cudaMemcpyDeviceToHost, m->stream));
    tr.mark("all enqueued", 0, nullptr);
    B2S_CUDA(cudaStreamSynchronize(m->stream));
    tr.mark("synchronized", 0, nullptr);
    if (batch_rejected(cnt)) {
        // every chunk is still in m->d_in: one launch over the whole batch takes it back out
        if ((rc = db.raycast(m, 0, scans, -1, nullptr, m->stream, true))) return rc;
        if (pmap_out) {
            rc = b2s_grid_finalize(m->hit, m->miss, m->xw, m->yw, m->w_hit, m->w_miss, m->thresh, nullptr,
                                   (int8_t *)m->d_pmap.p, m->stream);
            if (rc) return rc;
            B2S_CUDA(cudaMemcpyAsync(pmap_out, m->d_pmap.p, cells, cudaMemcpyDeviceToHost, m->stream));
        }
        B2S_CUDA(cudaStreamSynchronize(m->stream));
        return batch_error(cnt);
    }
    return B2S_OK;
}
}  // namespace

extern "C" int b2s_mapping_update(b2s_mapping *m, const float *ox, const float *oy, const float *cx,
                                  const float *cy, int scans, int beams, int8_t *pmap_out)
{
    B2S_REQUIRE(m, "b2s_mapping_update: null handle");
    B2S_REQUIRE(scans >= 0 && beams >= 0, "b2s_mapping_update: negative count");
    B2S_REQUIRE((size_t)scans * beams == 0 || (ox && oy && cx && cy), "b2s_mapping_update: null pointer");
    HostBatch hb = {false, false, ox, oy, cx, cy, nullptr, nullptr, nullptr, 0.0, nullptr};
    return mapping_update_impl(m, hb, scans, beams, pmap_out);
}

extern "C" int b2s_mapping_update_f64(b2s_mapping *m, const double *ox, const double *oy, const double *cx,
                                      const double *cy, int scans, int beams, int8_t *pmap_out)
{
    B2S_REQUIRE(m, "b2s_mapping_update_f64: null handle");
    B2S_REQUIRE(scans >= 0 && beams >= 0, "b2s_mapping_update_f64: negative count");
    B2S_REQUIRE((size_t)scans * beams == 0 || (ox && oy && cx && cy), "b2s_mapping_update_f64: null pointer");
    HostBatch hb = {false, true, ox, oy, cx, cy, nullptr, nullptr, nullptr, 0.0, nullptr};
    return mapping_update_impl(m, hb, scans, beams, pmap_out);
}

extern "C" int b2s_mapping_update_incremental(b2s_mapping *m, const float *ox, const float *oy, const float *cx,
                                              const float *cy, int scans, int beams, int8_t *pmap_inout,
                                              int32_t *tiles_out, int tiles_cap, int *tiles_count)
{
    B2S_REQUIRE(m && pmap_inout, "b2s_mapping_update_incremental: null pointer");
    B2S_REQUIRE(scans >= 0 && beams >= 0 && tiles_cap >= 0, "b2s_mapping_update_incremental: negative count");
    B2S_REQUIRE((size_t)scans * beams == 0 || (ox && oy && cx && cy), "b2s_mapping_update_incremental: null pointer");
    HostBatch hb = {false, false, ox, oy, cx, cy, nullptr, nullptr, nullptr, 0.0, nullptr};
    return mapping_update_impl(m, hb, scans, beams, pmap_inout, true, tiles_out, tiles_cap, tiles_count);
}

extern "C" int b2s_mapping_update_incremental_f64(b2s_mapping *m, const double *ox, const double *oy, const double *cx,
                                                  const double *cy, int scans, int beams, int8_t *pmap_inout,
                                                  int32_t *tiles_out, int tiles_cap, int *tiles_count)
{
    B2S_REQUIRE(m && pmap_inout, "b2s_mapping_update_incremental_f64: null pointer");
    B2S_REQUIRE(scans >= 0 && beams >= 0 && tiles_cap >= 0, "b2s_mapping_update_incremental_f64: negative count");
    B2S_REQUIRE((size_t)scans * beams == 0 || (ox && oy && cx && cy), "b2s_mapping_update_incremental_f64: null pointer");
    HostBatch hb = {false, true, ox, oy, cx, cy, nullptr, nullptr, nullptr, 0.0, nullptr};
    return mapping_update_impl(m, hb, scans, beams, pmap_inout, true, tiles_out, tiles_cap, tiles_count);
}

extern "C" int b2s_mapping_update_ranges(b2s_mapping *m, const float *ranges, const double *pose4,
                                         const double *beam_cs, double clamp_inf_to, int scans, int beams,
                                         int8_t *pmap_out)
{
    B2S_REQUIRE(m, "b2s_mapping_update_ranges: null handle");
    B2S_REQUIRE(scans >= 0 && beams >= 0, "b2s_mapping_update_ranges: negative count");
    B2S_REQUIRE((size_t)scans * beams == 0 || (ranges && pose4 && beam_cs), "b2s_mapping_update_ranges: null pointer");
    HostBatch hb = {true, false, nullptr, nullptr, nullptr, nullptr, ranges, pose4, beam_cs, clamp_inf_to, nullptr};
    return mapping_update_impl(m, hb, scans, beams, pmap_out);
}

extern "C" int b2s_mapping_update_scans(b2s_mapping *m, const float *ranges, const double *poses3,
                                        const double *beam_cs, double clamp_inf_to, int scans, int beams,
                                        int8_t *pmap_out)
{
    B2S_REQUIRE(m, "b2s_mapping_update_scans: null handle");
    B2S_REQUIRE(scans >= 0 && beams >= 0, "b2s_mapping_update_scans: negative count");
    B2S_REQUIRE((size_t)scans * beams == 0 || (ranges && poses3 && beam_cs), "b2s_mapping_update_scans: null pointer");
    HostBatch hb = {true, false, nullptr, nullptr, nullptr, nullptr, ranges, nullptr, beam_cs, clamp_inf_to, poses3};
    return mapping_update_impl(m, hb, scans, beams, pmap_out);
}

// ------------------------------------------------------------------------------ streaming Mapping calls
//
// b2s_mapping_update* are blocking: upload, ray-cast, finalize, read the map back, return.  Back to back they leave
// the copy engines idle while the kernels run and the SMs idle while the 16.8 MB map crosses PCIe.  The submit / wait
// pair keeps two steps in flight instead: submit enqueues a whole step (its own device input buffers, counters and
// device copy of the occupancy) and returns; the upload of step k + 1 then overlaps the ray-cast of step k and the
// read-back of step k - ... on a third stream.  wait(ticket) blocks until that step's map is in pmap_out and gives the
// step's verdict; a batch the reference would raise on is taken back out of the counts there (one sign -1 ray-cast of
// the slot's still-resident inputs: exact), but maps of steps submitted in between were finalized with it still applied.
namespace {
int mapping_wait_slot(b2s_mapping *m, MappingSlot &sl)
{
    if (!sl.in_flight) return B2S_OK;
    B2S_CUDA(cudaEventSynchronize(sl.done));
    sl.in_flight = false;
    if (!batch_rejected(sl.h_cnt)) return B2S_OK;
    // roll the step back: the inputs are still in the slot's device buffers (the slot is not reused before its wait)
    int rc = sl.batch.raycast(m, 0, sl.batch.scans, -1, nullptr, m->stream, true);
    if (rc) return rc;
    B2S_CUDA(cudaStreamSynchronize(m->stream));
    return batch_error(sl.h_cnt);
}

int mapping_submit_impl(b2s_mapping *m, const HostBatch &hb, int scans, int beams, int zero_first, int8_t *pmap_out,
                        int *ticket_out)
{
    DeviceGuard g(m->device);
    const int ticket = m->submitted;
    MappingSlot &sl = m->slot[ticket & 1];
    MappingSlot &other = m->slot[(ticket & 1) ^ 1];
    int rc;
    if (sl.in_flight && (rc = mapping_wait_slot(m, sl))) return rc;  // its buffers are about to be reused
    const size_t total = (size_t)scans * beams, cells = (size_t)m->xw * m->yw;
    const size_t poses = (size_t)scans * 4 * sizeof(double);
    DeviceBatch db(hb, scans, beams);
    if ((rc = sl.d_in.reserve(db.bytes()))) return rc;
    if ((rc = sl.d_map.reserve(cells))) return rc;
    if (hb.fused && hb.poses3 && (rc = sl.h_pose.reserve(poses ? poses : 16))) return rc;
    db.bind(sl.d_in.p);
    cudaStream_t cs = m->copy_stream;
    // the copy stream may overwrite the slot's inputs once the ray-casts that last read them are done
    B2S_CUDA(cudaStreamWaitEvent(cs, sl.inputs_free, 0));
    B2S_CUDA(cudaMemsetAsync(sl.d_cnt, 0, B2S_CNT_WORDS * sizeof(int32_t), m->stream));
    if (zero_first) {
        const size_t plane = cells * sizeof(int32_t);
        B2S_CUDA(cudaMemsetAsync(m->hit, 0, plane, m->stream));
        B2S_CUDA(cudaMemsetAsync(m->miss, 0, plane, m->stream));
    }
    if (total > 0) {
        // a step submitted while the other slot is in flight has its upload hidden under that step's ray-cast and
        // goes as one launch; a step that starts on an idle device is cut into ~1 M-beam chunks (see the blocking call)
        const int nchunk = pipeline_chunks(other.in_flight ? 1 : (int)((total + (1u << 20) - 1) >> 20), MAX_CHUNKS, scans);
        for (int k = 0; k < nchunk; ++k) {
            const size_t s0 = (size_t)scans * k / nchunk, s1 = (size_t)scans * (k + 1) / nchunk;
            if ((rc = db.upload(hb, s0, s1, (double *)sl.h_pose.p, cs))) return rc;
            B2S_CUDA(cudaEventRecord(m->chunk_ready[k], cs));
            B2S_CUDA(cudaStreamWaitEvent(m->stream, m->chunk_ready[k], 0));
            if ((rc = db.raycast(m, s0, s1, +1, sl.d_cnt, m->stream, k == nchunk - 1))) return rc;
        }
    }
    B2S_CUDA(cudaEventRecord(sl.inputs_free, m->stream));
    if (pmap_out) {
        rc = b2s_grid_finalize(m->hit, m->miss, m->xw, m->yw, m->w_hit, m->w_miss, m->thresh, nullptr, (int8_t *)sl.d_map.p,
                               m->stream);
        if (rc) return rc;
    }
    B2S_CUDA(cudaEventRecord(m->handoff, m->stream));
    B2S_CUDA(cudaStreamWaitEvent(m->d2h_stream, m->handoff, 0));
    if (pmap_out) B2S_CUDA(cudaMemcpyAsync(pmap_out, sl.d_map.p, cells, cudaMemcpyDeviceToHost, m->d2h_stream));
    B2S_CUDA(cudaMemcpyAsync(sl.h_cnt, sl.d_cnt, B2S_CNT_WORDS * sizeof(int32_t), cudaMemcpyDeviceToHost, m->d2h_stream));
    B2S_CUDA(cudaEventRecord(sl.done, m->d2h_stream));
    sl.in_flight = true;
    sl.ticket = ticket;
    sl.batch = db;
    m->pmap_valid = false;  // the incremental read-back of update() starts over after streamed steps
    m->submitted = ticket + 1;
    if (ticket_out) *ticket_out = ticket;
    return B2S_OK;
}
}  // namespace

extern "C" int b2s_mapping_submit(b2s_mapping *m, const float *ox, const float *oy, const float *cx, const float *cy,
                                  int scans, int beams, int zero_first, int8_t *pmap_out, int *ticket_out)
{
    B2S_REQUIRE(m && ticket_out, "b2s_mapping_submit: null pointer");
    B2S_REQUIRE(scans >= 0 && beams >= 0, "b2s_mapping_submit: negative count");
    B2S_REQUIRE((size_t)scans * beams == 0 || (ox && oy && cx && cy), "b2s_mapping_submit: null pointer");
    HostBatch hb = {false, false, ox, oy, cx, cy, nullptr, nullptr, nullptr, 0.0, nullptr};
    return mapping_submit_impl(m, hb, scans, beams, zero_first, pmap_out, ticket_out);
}

extern "C" int b2s_mapping_submit_scans(b2s_mapping *m, const float *ranges, const double *poses3, const double *beam_cs,
                                        double clamp_inf_to, int scans, int beams, int zero_first, int8_t *pmap_out,
                                        int *ticket_out)
{
    B2S_REQUIRE(m && ticket_out, "b2s_mapping_submit_scans: null pointer");
    B2S_REQUIRE(scans >= 0 && beams >= 0, "b2s_mapping_submit_scans: negative count");
    B2S_REQUIRE((size_t)scans * beams == 0 || (ranges && poses3 && beam_cs), "b2s_mapping_submit_scans: null pointer");
    HostBatch hb = {true, false, nullptr, nullptr, nullptr, nullptr, ranges, nullptr, beam_cs, clamp_inf_to, poses3};
    return mapping_submit_impl(m, hb, scans, beams, zero_first, pmap_out, ticket_out);
}

extern "C" int b2s_mapping_wait(b2s_mapping *m, int ticket)
{
    B2S_REQUIRE(m, "b2s_mapping_wait: null handle");
    B2S_REQUIRE(ticket >= 0 && ticket < m->submitted, "b2s_mapping_wait: unknown ticket");
    DeviceGuard g(m->device);
    MappingSlot &sl = m->slot[ticket & 1];
    if (!sl.in_flight || sl.ticket != ticket) return B2S_OK;  // already waited for (or superseded and waited implicitly)
    return mapping_wait_slot(m, sl);
}

extern "C" int b2s_mapping_read(b2s_mapping *m, int32_t *hit, int32_t *miss, float *datamap, int8_t *pmap)
{
    B2S_REQUIRE(m, "b2s_mapping_read: null handle");
    DeviceGuard g(m->device);
    const size_t cells = (size_t)m->xw * m->yw;
    int rc;
    if (datamap || pmap) {
        if (datamap && (rc = m->d_datamap.reserve(cells * sizeof(float)))) return rc;
        if (pmap && (rc = m->d_pmap.reserve(cells))) return rc;
        rc = b2s_grid_finalize(m->hit, m->miss, m->xw, m->yw, m->w_hit, m->w_miss, m->thresh,
                               datamap ? (float *)m->d_datamap.p : nullptr,
                               pmap ? (int8_t *)m->d_pmap.p : nullptr, m->stream);
        if (rc) return rc;
        if (datamap)
            B2S_CUDA(cudaMemcpyAsync(datamap, m->d_datamap.p, cells * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
        if (pmap) B2S_CUDA(cudaMemcpyAsync(pmap, m->d_pmap.p, cells, cudaMemcpyDeviceToHost, m->stream));
    }
    if (hit) B2S_CUDA(cudaMemcpyAsync(hit, m->hit, cells * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
    if (miss) B2S_CUDA(cudaMemcpyAsync(miss, m->miss, cells * sizeof(int32_t), cudaMemcpyDeviceToHost, m->stream));
    B2S_CUDA(cudaStreamSynchronize(m->stream));
    return B2S_OK;
}

extern "C" int b2s_mapping_write(b2s_mapping *m, const int32_t *hit, const int32_t *miss)
{
    B2S_REQUIRE(m && hit && miss, "b2s_mapping_write: null pointer");
    DeviceGuard g(m->device);
    const size_t plane = (size_t)m->xw * m->yw * sizeof(int32_t);
    B2S_CUDA(cudaMemcpyAsync(m->hit, hit, plane, cudaMemcpyHostToDevice, m->stream));
    B2S_CUDA(cudaMemcpyAsync(m->miss, miss, plane, cudaMemcpyHostToDevice, m->stream));
    B2S_CUDA(cudaStreamSynchronize(m->stream));
    m->pmap_valid = false;
    return B2S_OK;
}

extern "C" int b2s_mapping_planes(b2s_mapping *m, int32_t **hit, int32_t **miss, void **stream)
{
    B2S_REQUIRE(m, "b2s_mapping_planes: null handle");
    m->pmap_valid = false;  // the caller may change the planes behind the object's back: next read-back is a full one
    if (hit) *hit = m->hit;
    if (miss) *miss = m->miss;
    if (stream) *stream = (void *)m->stream;
    return B2S_OK;
}

extern "C" int b2s_bresenham_host(const int32_t *segs, int count, const int64_t *offsets, int32_t *cells_xy)
{
    B2S_REQUIRE(count >= 0, "b2s_bresenham_host: negative count");
    if (count == 0) return B2S_OK;
    B2S_REQUIRE(segs && offsets, "b2s_bresenham_host: null pointer");
    const int64_t total = offsets[count];
    B2S_REQUIRE(total >= 0 && (total == 0 || cells_xy), "b2s_bresenham_host: bad offsets");
    ScratchPool *sp = scratch_pool();
    if (!sp) return cuda_fail(cudaErrorUnknown, "b2s_bresenham_host: no device");
    int rc;
    if ((rc = sp->a.reserve((size_t)count * 16))) return rc;
    if ((rc = sp->b.reserve((size_t)(count + 1) * 8))) return rc;
    if ((rc = sp->c.reserve((size_t)(total > 0 ? total : 1) * 8))) return rc;
    B2S_CUDA(cudaMemcpyAsync(sp->a.p, segs, (size_t)count * 16, cudaMemcpyHostToDevice, cudaStreamPerThread));
    B2S_CUDA(cudaMemcpyAsync(sp->b.p, offsets, (size_t)(count + 1) * 8, cudaMemcpyHostToDevice, cudaStreamPerThread));
    if ((rc = b2s_bresenham_paths((const int32_t *)sp->a.p, count, (const int64_t *)sp->b.p, (int32_t *)sp->c.p,
                                  cudaStreamPerThread)))
        return rc;
    if (total > 0)
        B2S_CUDA(cudaMemcpyAsync(cells_xy, sp->c.p, (size_t)total * 8, cudaMemcpyDeviceToHost, cudaStreamPerThread));
    B2S_CUDA(cudaStreamSynchronize(cudaStreamPerThread));
    return B2S_OK;
}

// ------------------------------------------------------------------------------ NCCL (dlopen)
//
// The library is not linked against NCCL: in a torch process libnccl.so.2 is already loaded
// (torch bundles it) and dlopen returns that copy, so both sides share one NCCL runtime.

namespace {
typedef struct { char internal[128]; } nccl_uid;
typedef int (*fn_get_uid)(nccl_uid *);
typedef int (*fn_init_rank)(void **, int, nccl_uid, int);
typedef int (*fn_destroy)(void *);
typedef int (*fn_allreduce)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_group)(void);
typedef const char *(*fn_errstr)(int);

struct NcclApi {
    void *handle = nullptr;
    fn_get_uid get_uid = nullptr;
    fn_init_rank init_rank = nullptr;
    fn_destroy destroy = nullptr;
    fn_allreduce allreduce = nullptr;
    fn_group group_start = nullptr, group_end = nullptr;
    fn_errstr errstr = nullptr;
    bool tried = false;
};
NcclApi g_nccl;

int nccl_load()
{
    if (g_nccl.allreduce) return B2S_OK;
    if (!g_nccl.tried) {
        g_nccl.tried = true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *nm : names) {
            g_nccl.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (g_nccl.handle) break;
        }
        if (g_nccl.handle) {
            g_nccl.get_uid = (fn_get_uid)dlsym(g_nccl.handle, "ncclGetUniqueId");
            g_nccl.init_rank = (fn_init_rank)dlsym(g_nccl.handle, "ncclCommInitRank");
            g_nccl.destroy = (fn_destroy)dlsym(g_nccl.handle, "ncclCommDestroy");
            g_nccl.allreduce = (fn_allreduce)dlsym(g_nccl.handle, "ncclAllReduce");
            g_nccl.group_start = (fn_group)dlsym(g_nccl.handle, "ncclGroupStart");
            g_nccl.group_end = (fn_group)dlsym(g_nccl.handle, "ncclGroupEnd");
            g_nccl.errstr = (fn_errstr)dlsym(g_nccl.handle, "ncclGetErrorString");
        }
    }
    if (!g_nccl.allreduce || !g_nccl.get_uid || !g_nccl.init_rank || !g_nccl.destroy || !g_nccl.group_start ||
        !g_nccl.group_end) {
        set_error("NCCL not available: %s", g_nccl.handle ? "missing symbols" : "libnccl.so.2 not found");
        return B2S_ERR_NCCL;
    }
    return B2S_OK;
}

int nccl_fail(int code, const char *what)
{
    set_error("%s: %s", what, g_nccl.errstr ? g_nccl.errstr(code) : "nccl error");
    return B2S_ERR_NCCL;
}
}  // namespace

extern "C" int b2s_nccl_unique_id(void *id128)
{
    B2S_REQUIRE(id128, "b2s_nccl_unique_id: null pointer");
    int rc = nccl_load();
    if (rc) return rc;
    nccl_uid uid;
    int e = g_nccl.get_uid(&uid);
    if (e) return nccl_fail(e, "ncclGetUniqueId");
    memcpy(id128, &uid, sizeof(uid));
    return B2S_OK;
}

extern "C" int b2s_nccl_comm_init(void **comm_out, int nranks, int rank, const void *id128)
{
    B2S_REQUIRE(comm_out && id128 && nranks > 0 && rank >= 0 && rank < nranks, "b2s_nccl_comm_init: bad arguments");
    int rc = nccl_load();
    if (rc) return rc;
    nccl_uid uid;
    memcpy(&uid, id128, sizeof(uid));
    int e = g_nccl.init_rank(comm_out, nranks, uid, rank);
    if (e) return nccl_fail(e, "ncclCommInitRank");
    return B2S_OK;
}

extern "C" int b2s_nccl_comm_destroy(void *comm)
{
    if (!comm) return B2S_OK;
    int rc = nccl_load();
    if (rc) return rc;
    int e = g_nccl.destroy(comm);
    if (e) return nccl_fail(e, "ncclCommDestroy");
    return B2S_OK;
}

extern "C" int b2s_grid_allreduce(int32_t *hit, int32_t *miss, size_t cells, void *nccl_comm, void *stream)
{
    B2S_REQUIRE(hit && miss && nccl_comm, "b2s_grid_allreduce: null pointer");
    int rc = nccl_load();
    if (rc) return rc;
    const int nccl_int32 = 2, nccl_sum = 0;  // ncclInt32, ncclSum
    int e = g_nccl.group_start();
    if (e) return nccl_fail(e, "ncclGroupStart");
    e = g_nccl.allreduce(hit, hit, cells, nccl_int32, nccl_sum, nccl_comm, (cudaStream_t)stream);
    if (!e) e = g_nccl.allreduce(miss, miss, cells, nccl_int32, nccl_sum, nccl_comm, (cudaStream_t)stream);
    int e2 = g_nccl.group_end();
    if (e) return nccl_fail(e, "ncclAllReduce");
    if (e2) return nccl_fail(e2, "ncclGroupEnd");
    return B2S_OK;
}
