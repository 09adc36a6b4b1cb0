// Microbenchmark for an env-step made of short-lived work items (DESIGN §4): does a launch whose warps each take ONE item
// from a ticket -- a rule item (the rule work of a 32-env tile, then "tile complete" on the tile's word) or a row item (wait
// for its tile's word, then write a slice of the tile's thermometer rows and exit) -- stream rows faster than k_env's one
// wave of long-lived warps?
//
// Rule items are synthetic: each spins for its tile's lifetime, drawn from the rule-kernel trace of the split experiment
// (profiles/r2x_split_row_writer_experiment.json: p50 20 us, p99 36 us, max 49 us), and writes 8 KB of state and packed list.
// Row items read 16-byte row descriptors (what face_planes leaves in shared memory) and write 240-byte rows into
// compressible memory, lanes 0..29 = (row parity, rank) as in k_env.  Per tile: 288 face rows (32 envs x 9 planes) and
// 100..259 action rows (mean 180, N = 5.6 moves per env).  Ticket order: the first LAG tickets are rule items, then every
// period is [the FS-env face slices and the action item of tile s, rule item of tile s + LAG].
// The baseline is k_env's shape in the same call: one wave of 2-warp CTAs, each warp spins its tile's lifetime in two parts
// and writes the same rows in k_env's phase order (even tiles face rows before the second part, odd tiles after).
// Both run as one launch of 4096 tiles (131 072 envs) and as four concurrent streams of 1024 tiles (bench.py config 4).
// Occupancy is pinned to k_env's 28 warps per SM with 7 296 B of shared memory per warp.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o row_items row_items.cu -lcuda
#include <cuda.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); exit(1); } } while (0)
#define CU(x) do { CUresult e = (x); if (e != CUDA_SUCCESS) { const char* s; cuGetErrorString(e, &s); printf("driver error %s at %d\n", s, __LINE__); exit(1); } } while (0)

constexpr int kFaceRows = 288, kSmemPerWarp = 7296;
struct __align__(16) Desc { unsigned lo, hi; float s, pad; };
struct Tiles {   // one launch's tiles
    const Desc* desc; const long long* act_off; const int* life_ns; float4* face; float4* act; float4* scratch;
    unsigned long long* word; unsigned* ticket; int nt;
};

__global__ void k_fill_desc(Desc* d, size_t nrows, unsigned seed) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrows) return;
    unsigned x = seed ^ (unsigned)(i * 2654435761u), lo = 0, hi = 0;
    for (int k = 0; k < 15; k++) {
        x = x * 1664525u + 1013904223u;
        const unsigned c = (x >> 24) % 9 < 5 ? 0u : ((x >> 16) & 3u) + 1u;
        if (k < 8) lo |= c << (4 * k); else hi |= c << (4 * (k - 8));
    }
    Desc v; v.lo = lo; v.hi = hi; v.s = (i % 9 >= 7) ? 0.4375f : 1.f; v.pad = 0.f;
    d[i] = v;
}

__device__ __forceinline__ unsigned long long now_ns() {
    unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t;
}
__device__ __forceinline__ void spin(long long ns) {   // busy, like rule work: it takes issue slots
    const unsigned long long t0 = now_ns();
    while ((long long)(now_ns() - t0) < ns) {}
}
__device__ __forceinline__ void rows(float4* gdst, const Desc* __restrict__ d, int nrows, int lane, const float4* lut) {
    if (lane >= 30) return;
    const int k = lane % 15;
    float4* dst = gdst + lane;
#pragma unroll 4
    for (int r = lane / 15; r < nrows; r += 2, dst += 30) {
        const Desc v = d[r];
        float4 q = lut[((k < 8 ? v.lo : v.hi) >> (4 * (k & 7))) & 15u];
        q.x *= v.s; q.y *= v.s; q.z *= v.s; q.w *= v.s;
        __stcs(dst, q);
    }
}
__device__ __forceinline__ void state_stores(const Tiles& T, int t, int lane) {   // 8 KB: state, packed list, offsets
    float4* p = T.scratch + (size_t)t * 512 + lane;
#pragma unroll
    for (int i = 0; i < 16; i++) p[32 * i] = make_float4((float)t, 0.f, 0.f, 0.f);
}
__device__ __forceinline__ void act_rows(const Tiles& T, int t, int lane, const float4* lut) {
    const long long a0 = T.act_off[t], n = T.act_off[t + 1] - a0;
    rows(T.act + a0 * 15, T.desc + (size_t)t * kFaceRows, (int)n, lane, lut);   // descriptors: any L2-resident 16 B rows
}

template <int W>
__global__ void __launch_bounds__(32 * W) k_wave(Tiles T) {   // k_env's shape: warp = tile, one wave, static ids
    extern __shared__ float4 lut_raw[];
    float4* lut = lut_raw + 16 * (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31, t = blockIdx.x * W + (threadIdx.x >> 5);
    if (lane < 16) lut[lane] = make_float4(lane > 0 && lane < 8, lane > 1 && lane < 8, lane > 2 && lane < 8, lane > 3 && lane < 8);
    __syncwarp();
    if (t >= T.nt) return;
    const int life = T.life_ns[t];
    spin(life * 2 / 5);
    state_stores(T, t, lane);
    if (t & 1) spin(life - life * 2 / 5);
    rows(T.face + (size_t)t * kFaceRows * 15, T.desc + (size_t)t * kFaceRows, kFaceRows, lane, lut);
    if (!(t & 1)) spin(life - life * 2 / 5);
    act_rows(T, t, lane, lut);
}

template <int W, int FS, int LAG>
__global__ void __launch_bounds__(32 * W) k_items(Tiles T, unsigned long long epoch_tag, unsigned* poll_fail) {
    constexpr int R = 32 / FS + 1;   // row items per tile: the face slices, then the action rows
    extern __shared__ float4 lut_raw[];
    float4* lut = lut_raw + 16 * (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (lane < 16) lut[lane] = make_float4(lane > 0 && lane < 8, lane > 1 && lane < 8, lane > 2 && lane < 8, lane > 3 && lane < 8);
    int i = 0;
    if (lane == 0) i = (int)atomicAdd(T.ticket, 1u);
    i = __shfl_sync(0xFFFFFFFFu, i, 0);
    __syncwarp();
    const int nt = T.nt, lag = LAG < nt ? LAG : nt;
    int t, j;   // j == R: rule item
    if (i < lag) { t = i; j = R; }
    else {
        const int i2 = i - lag;
        if (i2 < (nt - lag) * (R + 1)) { const int s = i2 / (R + 1); j = i2 % (R + 1); t = j == R ? s + lag : s; }
        else { const int i3 = i2 - (nt - lag) * (R + 1); t = nt - lag + i3 / R; j = i3 % R; }
    }
    if (t >= nt) return;
    if (j == R) {
        spin(T.life_ns[t]);
        state_stores(T, t, lane);
        __threadfence();
        if (lane == 0) asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(T.word + t), "l"(epoch_tag | (3ull << 32)) : "memory");
        return;
    }
    unsigned spins = 0;
    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(T.word + t) : "memory");
        w = __shfl_sync(0xFFFFFFFFu, w, 0);
        if ((w >> 34) == (epoch_tag >> 34) && ((w >> 32) & 3ull) == 3ull) break;
        __nanosleep(128);
        if (++spins > (1u << 22)) { if (lane == 0) atomicAdd(poll_fail, 1u); return; }
    }
    if (j < R - 1) {
        const size_t r0 = (size_t)t * kFaceRows + (size_t)j * FS * 9;
        rows(T.face + r0 * 15, T.desc + r0, FS * 9, lane, lut);
    } else {
        act_rows(T, t, lane, lut);
    }
}

static float4* alloc_vmm(size_t bytes) {
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = 0;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    CU(cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
    const size_t size = (bytes + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle h;
    CU(cuMemCreate(&h, size, &prop, 0));
    CUdeviceptr p;
    CU(cuMemAddressReserve(&p, size, 0, 0, 0));
    CU(cuMemMap(p, size, 0, h, 0));
    CUmemAccessDesc acc = {};
    acc.location = prop.location; acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    CU(cuMemSetAccess(p, size, &acc, 1));
    return (float4*)p;
}

constexpr int kTilesTotal = 4096, kIters = 40;
static Tiles g_tiles[4];
static unsigned* g_tickets;   // [kIters + warm-up][4]
static unsigned* g_fail;
static double g_row_bytes;
static cudaStream_t g_st[4];
static unsigned long long g_epoch = 0;   // tile words are never cleared: every launch has its own epoch

// ms per step (all 4096 tiles) over kIters steps, after 4 warm-up steps; launch(step, group, stream) enqueues one launch
template <class F> static double time_steps(int groups, F launch) {
    cudaEvent_t a, b, done[4];
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    for (int g = 0; g < 4; g++) CK(cudaEventCreate(&done[g]));
    CK(cudaMemset(g_tickets, 0, sizeof(unsigned) * (kIters + 4) * 4));
    CK(cudaDeviceSynchronize());
    for (int it = 0; it < kIters + 4; it++) {
        if (it == 4) { CK(cudaEventRecord(a, g_st[0])); for (int g = 1; g < groups; g++) CK(cudaStreamWaitEvent(g_st[g], a)); }
        for (int g = 0; g < groups; g++) launch(it, g, g_st[g]);
    }
    for (int g = 1; g < groups; g++) { CK(cudaEventRecord(done[g], g_st[g])); CK(cudaStreamWaitEvent(g_st[0], done[g])); }
    CK(cudaEventRecord(b, g_st[0]));
    CK(cudaEventSynchronize(b));
    CK(cudaGetLastError());
    float ms; CK(cudaEventElapsedTime(&ms, a, b));
    return ms / kIters;
}

static void report(const char* name, double ms) {
    printf(", \"%s_ms\": %.4f, \"%s_row_TBs\": %.3f", name, ms, name, g_row_bytes / ms / 1e9);
    fflush(stdout);
}

template <int W> static void wave(int groups, const char* name) {
    const int per = kTilesTotal / groups, grid = (per + W - 1) / W;
    const size_t smem = (size_t)W * kSmemPerWarp;
    CK(cudaFuncSetAttribute(k_wave<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    report(name, time_steps(groups, [&](int, int g, cudaStream_t st) { k_wave<W><<<grid, 32 * W, smem, st>>>(g_tiles[g]); }));
}
template <int W, int FS, int LAG> static void items(int groups, const char* name) {
    const int per = kTilesTotal / groups, nitems = per * (32 / FS + 2), grid = (nitems + W - 1) / W;
    const size_t smem = (size_t)W * kSmemPerWarp;
    CK(cudaFuncSetAttribute(k_items<W, FS, LAG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    report(name, time_steps(groups, [&](int it, int g, cudaStream_t st) {
        Tiles T = g_tiles[g]; T.ticket = g_tickets + it * 4 + g;
        k_items<W, FS, LAG><<<grid, 32 * W, smem, st>>>(T, (g_epoch + it + 1) << 34, g_fail);
    }));
    g_epoch += kIters + 4;
}

int main() {
    CK(cudaFree(0));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, 0));
    // lifetimes: log-normal with median 20 us and p99 36 us (sigma = ln(1.8) / 2.326), cut at 49 us
    std::vector<int> life(kTilesTotal);
    std::vector<long long> off(kTilesTotal + 1, 0);
    unsigned x = 12345u;
    auto u01 = [&] { x = x * 1664525u + 1013904223u; return ((x >> 8) + 0.5) / 16777216.0; };
    for (int t = 0; t < kTilesTotal; t++) {
        const double z = std::sqrt(-2.0 * std::log(u01())) * std::cos(6.283185307179586 * u01());
        life[t] = (int)std::min(49000.0, 20000.0 * std::exp(z * std::log(1.8) / 2.326));
        off[t + 1] = off[t] + 100 + (long long)(u01() * 160);
    }
    std::vector<int> sorted(life); std::sort(sorted.begin(), sorted.end());
    const double face_rows = (double)kTilesTotal * kFaceRows, act_rows_n = (double)off[kTilesTotal];
    g_row_bytes = (face_rows + act_rows_n) * 240.0;
    printf("{\"device\": \"%s\", \"sms\": %d, \"tiles\": %d, \"row_bytes\": %.0f, \"face_rows\": %.0f, \"action_rows\": %.0f, "
           "\"life_us_p50\": %.1f, \"life_us_p99\": %.1f, \"life_us_max\": %.1f",
           prop.name, prop.multiProcessorCount, kTilesTotal, g_row_bytes, face_rows, act_rows_n,
           sorted[kTilesTotal / 2] / 1e3, sorted[kTilesTotal * 99 / 100] / 1e3, sorted.back() / 1e3);

    Desc* desc; CK(cudaMalloc(&desc, face_rows * sizeof(Desc)));
    k_fill_desc<<<(unsigned)((face_rows + 255) / 256), 256>>>(desc, (size_t)face_rows, 3u);
    int* life_d; long long* off_d; float4* scratch; unsigned long long* words;
    CK(cudaMalloc(&life_d, sizeof(int) * kTilesTotal));
    CK(cudaMalloc(&off_d, sizeof(long long) * (kTilesTotal + 4)));
    CK(cudaMalloc(&scratch, (size_t)kTilesTotal * 512 * sizeof(float4)));
    CK(cudaMalloc(&words, sizeof(unsigned long long) * kTilesTotal));
    CK(cudaMalloc(&g_tickets, sizeof(unsigned) * (kIters + 4) * 4));
    CK(cudaMalloc(&g_fail, sizeof(unsigned)));
    CK(cudaMemset(words, 0, sizeof(unsigned long long) * kTilesTotal));
    CK(cudaMemset(g_fail, 0, sizeof(unsigned)));
    CK(cudaMemcpy(life_d, life.data(), sizeof(int) * kTilesTotal, cudaMemcpyHostToDevice));
    float4* face = alloc_vmm((size_t)face_rows * 240);
    float4* act = alloc_vmm((size_t)act_rows_n * 240);
    for (int g = 0; g < 4; g++) CK(cudaStreamCreateWithFlags(&g_st[g], cudaStreamNonBlocking));

    for (int groups : {1, 4}) {
        const int per = kTilesTotal / groups;
        for (int g = 0; g < groups; g++) {   // group g = tiles [g * per, (g + 1) * per): its own offsets, words, rows
            std::vector<long long> o(per + 1);
            for (int t = 0; t <= per; t++) o[t] = off[g * per + t] - off[g * per];
            CK(cudaMemcpy(off_d + g * (per + 1), o.data(), sizeof(long long) * (per + 1), cudaMemcpyHostToDevice));
        }
        for (int g = 0; g < groups; g++) {
            Tiles& T = g_tiles[g];
            T.desc = desc + (size_t)g * per * kFaceRows; T.act_off = off_d + g * (per + 1); T.life_ns = life_d + g * per;
            T.face = face + (size_t)g * per * kFaceRows * 15; T.act = act + (size_t)off[g * per] * 15;
            T.scratch = scratch + (size_t)g * per * 512; T.word = words + g * per; T.ticket = nullptr; T.nt = per;
        }
        printf(", \"groups%d\": {\"x\": 0", groups);
        wave<2>(groups, "wave_kenv_shape");
        items<1, 8, 64>(groups, "items_fs8_lag64_w1");
        items<1, 8, 256>(groups, "items_fs8_lag256_w1");
        items<1, 8, 1024>(groups, "items_fs8_lag1024_w1");
        items<1, 16, 256>(groups, "items_fs16_lag256_w1");
        items<1, 32, 256>(groups, "items_fs32_lag256_w1");
        items<2, 8, 256>(groups, "items_fs8_lag256_w2");
        items<1, 4, 256>(groups, "items_fs4_lag256_w1");
        wave<2>(groups, "wave_kenv_shape_again");
        printf("}");
    }
    unsigned fail = 0; CK(cudaMemcpy(&fail, g_fail, sizeof fail, cudaMemcpyDeviceToHost));
    printf(", \"poll_timeouts\": %u}\n", fail);
    return 0;
}
