// Micro-benchmark behind DESIGN.md "why the grid kernel looks the way it does": sustained rate of the
// update primitives the ray-cast could use, on one B200.  Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3
//   redg32 / redg64 : red.global.add on spread addresses inside an L2-resident 64 MiB plane, A of 32 lanes active
//   atoms32         : atomicAdd on shared memory, spread addresses inside a 64 KiB tile
//   bulkred         : cp.reduce.async.bulk.global.shared::cta.add.s32 of ROW-byte rows (TMA reduce)
//   atoms_popc      : unpredicated atomicAdd(&smem, 1) (ATOMS.POPC.INC), L lanes per word
//   atoms_walk      : the same instruction from fanned-out "beams" walking a row-major tile, x-major or y-major,
//                     odd or even row pitch (bank conflicts of the y-major walk)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA %s at %d\n", cudaGetErrorString(e), __LINE__); exit(1); } } while (0)

__device__ __forceinline__ uint32_t lcg(uint32_t &s) { s = s * 1664525u + 1013904223u; return s; }

template <int ACTIVE, bool WIDE>
__global__ void __launch_bounds__(256) k_redg(int *plane, unsigned mask, int iters)
{
    uint32_t s = blockIdx.x * 256 + threadIdx.x + 1;
    const int lane = threadIdx.x & 31;
    // each warp walks a random column-like window: lanes hit consecutive words (like adjacent cells)
    for (int i = 0; i < iters; ++i) {
        uint32_t base = __shfl_sync(0xffffffffu, lcg(s), 0) & mask;
        if (lane < ACTIVE) {
            if (WIDE) atomicAdd(reinterpret_cast<unsigned long long *>(plane) + ((base >> 1) + lane), 0x100000001ull);
            else atomicAdd(plane + base + lane, 1);
        }
    }
}

// Runs of RUN adjacent lanes on the same word (what the ray-cast sees: adjacent beams share cells).  ALL = false:
// only the run heads issue the RED, with the run length (the kernel's scheme, a divergent branch around the RED).
// ALL = true: every lane issues it unconditionally, non-heads add 0 -- no branch, RUN times the lane-ops.
template <int RUN, bool ALL>
__global__ void __launch_bounds__(256) k_redg_runs(int *plane, unsigned mask, int iters)
{
    uint32_t s = blockIdx.x * 256 + threadIdx.x + 1;
    const int lane = threadIdx.x & 31;
    const bool head = (lane % RUN) == 0;
    for (int i = 0; i < iters; ++i) {
        uint32_t base = __shfl_sync(0xffffffffu, lcg(s), 0) & mask;
        int *p = plane + base + lane / RUN;
        if (ALL) asm volatile("red.global.add.s32 [%0], %1;" ::"l"(p), "r"(head ? RUN : 0) : "memory");
        else if (head) asm volatile("red.global.add.s32 [%0], %1;" ::"l"(p), "r"(RUN) : "memory");
    }
}

template <int ACTIVE>
__global__ void __launch_bounds__(256) k_redg_scatter(int *plane, unsigned mask, int iters)
{
    uint32_t s = blockIdx.x * 256 + threadIdx.x + 1;
    const int lane = threadIdx.x & 31;
    for (int i = 0; i < iters; ++i) {
        uint32_t a = lcg(s) & mask;  // every lane its own random word
        if (lane < ACTIVE) atomicAdd(plane + a, 1);
    }
}

template <int ACTIVE>
__global__ void __launch_bounds__(256) k_atoms(int *out, int iters)
{
    extern __shared__ int tile[];
    for (int i = threadIdx.x; i < 16384; i += 256) tile[i] = 0;
    __syncthreads();
    uint32_t s = blockIdx.x * 256 + threadIdx.x + 1;
    const int lane = threadIdx.x & 31;
    for (int i = 0; i < iters; ++i) {
        uint32_t base = __shfl_sync(0xffffffffu, lcg(s), 0) & 16383u;
        if (lane < ACTIVE) atomicAdd(&tile[(base + lane) & 16383], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) out[blockIdx.x] = tile[0];
}

template <int ACTIVE>
__global__ void __launch_bounds__(256) k_atoms_scatter(int *out, int iters)
{
    extern __shared__ int tile[];
    for (int i = threadIdx.x; i < 16384; i += 256) tile[i] = 0;
    __syncthreads();
    uint32_t s = blockIdx.x * 256 + threadIdx.x + 1;
    const int lane = threadIdx.x & 31;
    for (int i = 0; i < iters; ++i) {
        uint32_t a = lcg(s) & 16383u;
        if (lane < ACTIVE) atomicAdd(&tile[a], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) out[blockIdx.x] = tile[0];
}

// Unpredicated atomicAdd(&tile[w], 1) with an unused result compiles to ATOMS.POPC.INC (no divergent region).
// LPW adjacent lanes share one word; the warp's words are consecutive.
template <int LPW>
__global__ void __launch_bounds__(256) k_atoms_popc(int *out, int iters)
{
    extern __shared__ int tile[];
    for (int i = threadIdx.x; i < 16384; i += 256) tile[i] = 0;
    __syncthreads();
    uint32_t s = blockIdx.x * 256 + threadIdx.x + 1;
    const int lane = threadIdx.x & 31;
    for (int i = 0; i < iters; ++i) {
        uint32_t base = __shfl_sync(0xffffffffu, lcg(s), 0) & 16383u;
        atomicAdd(&tile[(base + lane / LPW) & 16383], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) out[blockIdx.x] = tile[0];
}

// 32 beams fanned out over 1/32 of a radian each, walked from a common origin in a row-major tile of PITCH words
// per row: at step i lane l sits (l * i) / 64 cells off the warp's common line.  X-major: the step moves along a
// row (+PITCH per step is the other axis: rows are x); Y-major: the step moves down the row, lanes spread over
// rows, so their words are PITCH apart -- an even pitch puts them in few banks.
template <bool YMAJOR, int PITCH>
__global__ void __launch_bounds__(256) k_atoms_walk(int *out, int iters)
{
    extern __shared__ int tile[];
    for (int i = threadIdx.x; i < PITCH * 160; i += 256) tile[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (int it = 0; it < iters; it += 128) {
        for (int i = 0; i < 128; ++i) {
            const int spread = (lane * i) >> 6;  // 0 .. 63
            const int x = YMAJOR ? spread : i, y = YMAJOR ? i : spread;
            atomicAdd(&tile[x * PITCH + y], 1);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) out[blockIdx.x] = tile[0];
}

// plain (non-atomic) shared-memory read-modify-write, for the ownership-based designs
__global__ void __launch_bounds__(256) k_smem_rmw(int *out, int iters)
{
    extern __shared__ int tile[];
    for (int i = threadIdx.x; i < 16384; i += 256) tile[i] = 0;
    __syncthreads();
    uint32_t s = blockIdx.x * 256 + threadIdx.x + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = 0; i < iters; ++i) {
        uint32_t base = __shfl_sync(0xffffffffu, lcg(s), 0) & 2047u;
        int *p = &tile[warp * 2048 + ((base + lane * 33) & 2047)];  // warp-private slab, conflict-free stride
        *p = *p + 1;
    }
    __syncthreads();
    if (threadIdx.x == 0) out[blockIdx.x] = tile[0];
}

template <int ROW>
__global__ void __launch_bounds__(256) k_bulkred(int *plane, unsigned mask, int iters)
{
    __shared__ __align__(128) int rows[8][ROW / 4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = lane; i < ROW / 4; i += 32) rows[warp][i] = 1;
    __syncthreads();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    uint32_t s = blockIdx.x * 256 + threadIdx.x + 1;
    for (int i = 0; i < iters; ++i) {
        uint32_t base = (__shfl_sync(0xffffffffu, lcg(s), 0) & mask) & ~3u;  // 16-byte aligned
        if (lane == 0) {
            asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.s32 [%0], [%1], %2;" ::"l"(plane + base),
                         "r"((uint32_t)__cvta_generic_to_shared(&rows[warp][0])), "r"(ROW)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            if ((i & 7) == 7) asm volatile("cp.async.bulk.wait_group.read 4;" ::: "memory");
        }
        __syncwarp();
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

template <typename F>
static float time_ms(F launch)
{
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    launch();
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(a));
    launch();
    CK(cudaEventRecord(b));
    CK(cudaEventSynchronize(b));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, a, b));
    return ms;
}

int main()
{
    const size_t words = 16u << 20;  // 64 MiB int32 plane (L2 resident)
    int *plane, *out;
    CK(cudaMalloc(&plane, words * 4 + 4096));
    CK(cudaMemset(plane, 0, words * 4 + 4096));
    CK(cudaMalloc(&out, 1 << 20));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    const int sms = prop.multiProcessorCount;
    const int blocks = sms * 8, iters = 2000;
    const unsigned mask = (unsigned)(words - 1);
    int khz = 0;
    CK(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, 0));
    const double clk = khz * 1e3;
    printf("device %s, %d SMs, %.0f MHz nominal\n", prop.name, sms, clk / 1e6);
#define REPORT(name, active, ms) printf("%-26s active=%2d  %8.3f ms  %7.2f Gops/s  %6.3f lane-ops/clk/SM  %6.2f clk per warp-instr per SM\n", \
        name, active, ms, (double)blocks * 8 * iters * active / (ms * 1e-3) / 1e9, \
        (double)blocks * 8 * iters * active / (ms * 1e-3) / clk / sms, (ms * 1e-3) * clk * sms / ((double)blocks * 8 * iters))
    float ms;
#define REPORT2(name, active, ms, it) printf("%-26s active=%2d  %8.3f ms  %7.2f Gops/s  %6.3f lane-ops/clk/SM  %6.2f clk per warp-instr per SM\n", \
        name, active, ms, (double)blocks * 8 * (it) * active / (ms * 1e-3) / 1e9, \
        (double)blocks * 8 * (it) * active / (ms * 1e-3) / clk / sms, (ms * 1e-3) * clk * sms / ((double)blocks * 8 * (it)))
    ms = time_ms([&] { k_redg<32, false><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 contiguous lanes", 32, ms);
    ms = time_ms([&] { k_redg<16, false><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 contiguous lanes", 16, ms);
    ms = time_ms([&] { k_redg<8, false><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 contiguous lanes", 8, ms);
    ms = time_ms([&] { k_redg<4, false><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 contiguous lanes", 4, ms);
    ms = time_ms([&] { k_redg<1, false><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 contiguous lanes", 1, ms);
    ms = time_ms([&] { k_redg<32, true><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg64 contiguous lanes", 32, ms);
    ms = time_ms([&] { k_redg<8, true><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg64 contiguous lanes", 8, ms);
    ms = time_ms([&] { k_redg<4, true><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg64 contiguous lanes", 4, ms);
    ms = time_ms([&] { k_redg_runs<4, false><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 runs of 4, heads only", 8, ms);
    ms = time_ms([&] { k_redg_runs<4, true><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 runs of 4, all lanes", 32, ms);
    ms = time_ms([&] { k_redg_runs<8, false><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 runs of 8, heads only", 4, ms);
    ms = time_ms([&] { k_redg_runs<8, true><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 runs of 8, all lanes", 32, ms);
    ms = time_ms([&] { k_redg_runs<2, false><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 runs of 2, heads only", 16, ms);
    ms = time_ms([&] { k_redg_runs<2, true><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 runs of 2, all lanes", 32, ms);
    ms = time_ms([&] { k_redg_scatter<32><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 scattered lanes", 32, ms);
    ms = time_ms([&] { k_redg_scatter<8><<<blocks, 256>>>(plane, mask, iters); }); REPORT("redg32 scattered lanes", 8, ms);
    CK(cudaFuncSetAttribute(k_atoms<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
    CK(cudaFuncSetAttribute(k_atoms<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
    CK(cudaFuncSetAttribute(k_atoms_scatter<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
    CK(cudaFuncSetAttribute(k_atoms_scatter<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
    CK(cudaFuncSetAttribute(k_smem_rmw, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
    ms = time_ms([&] { k_atoms<32><<<blocks, 256, 65536>>>(out, iters); }); REPORT("atoms32 contiguous lanes", 32, ms);
    ms = time_ms([&] { k_atoms<8><<<blocks, 256, 65536>>>(out, iters); }); REPORT("atoms32 contiguous lanes", 8, ms);
    ms = time_ms([&] { k_atoms_scatter<32><<<blocks, 256, 65536>>>(out, iters); }); REPORT("atoms32 scattered lanes", 32, ms);
    ms = time_ms([&] { k_atoms_scatter<8><<<blocks, 256, 65536>>>(out, iters); }); REPORT("atoms32 scattered lanes", 8, ms);
    ms = time_ms([&] { k_smem_rmw<<<blocks, 256, 65536>>>(out, iters); }); REPORT("smem ld+add+st (owned)", 32, ms);
    ms = time_ms([&] { k_bulkred<64><<<blocks, 256>>>(plane, mask, iters); }); REPORT("bulk reduce 64 B rows", 16, ms);
    ms = time_ms([&] { k_bulkred<128><<<blocks, 256>>>(plane, mask, iters); }); REPORT("bulk reduce 128 B rows", 32, ms);
    ms = time_ms([&] { k_bulkred<256><<<blocks, 256>>>(plane, mask, iters); }); REPORT("bulk reduce 256 B rows", 64, ms);
    {
        const int tile_bytes = 161 * 160 * 4;  // also holds PITCH = 160
        CK(cudaFuncSetAttribute(k_atoms_popc<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
        CK(cudaFuncSetAttribute(k_atoms_popc<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
        CK(cudaFuncSetAttribute(k_atoms_popc<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
        CK(cudaFuncSetAttribute(k_atoms_popc<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
        CK(cudaFuncSetAttribute(k_atoms_walk<false, 161>, cudaFuncAttributeMaxDynamicSharedMemorySize, tile_bytes));
        CK(cudaFuncSetAttribute(k_atoms_walk<true, 161>, cudaFuncAttributeMaxDynamicSharedMemorySize, tile_bytes));
        CK(cudaFuncSetAttribute(k_atoms_walk<false, 160>, cudaFuncAttributeMaxDynamicSharedMemorySize, tile_bytes));
        CK(cudaFuncSetAttribute(k_atoms_walk<true, 160>, cudaFuncAttributeMaxDynamicSharedMemorySize, tile_bytes));
        ms = time_ms([&] { k_atoms_popc<1><<<blocks, 256, 65536>>>(out, iters); }); REPORT("atoms.popc.inc 1 lane/word", 32, ms);
        ms = time_ms([&] { k_atoms_popc<2><<<blocks, 256, 65536>>>(out, iters); }); REPORT("atoms.popc.inc 2 lanes/word", 32, ms);
        ms = time_ms([&] { k_atoms_popc<4><<<blocks, 256, 65536>>>(out, iters); }); REPORT("atoms.popc.inc 4 lanes/word", 32, ms);
        ms = time_ms([&] { k_atoms_popc<32><<<blocks, 256, 65536>>>(out, iters); }); REPORT("atoms.popc.inc 32 lanes/word", 32, ms);
        const int wi = 2048;  // multiple of 128
        ms = time_ms([&] { k_atoms_walk<false, 161><<<blocks, 256, tile_bytes>>>(out, wi); }); REPORT2("walk x-major, pitch 161", 32, ms, wi);
        ms = time_ms([&] { k_atoms_walk<true, 161><<<blocks, 256, tile_bytes>>>(out, wi); }); REPORT2("walk y-major, pitch 161", 32, ms, wi);
        ms = time_ms([&] { k_atoms_walk<false, 160><<<blocks, 256, tile_bytes>>>(out, wi); }); REPORT2("walk x-major, pitch 160", 32, ms, wi);
        ms = time_ms([&] { k_atoms_walk<true, 160><<<blocks, 256, tile_bytes>>>(out, wi); }); REPORT2("walk y-major, pitch 160", 32, ms, wi);
    }
    return 0;
}
