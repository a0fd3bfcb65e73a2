// stream_mix.cu — microbenchmark (not product code): the streaming ceilings of the two SVGD kernels at n = 10, with
// the consumers laid out as in the product kernels.  One persistent CTA per SM, a producer warp filling a
// shared-memory ring, consumer warps reading every element of a stage before releasing it.
//   k1: read-only stream of [10 x 1024] tiles (K1's stage) through 2..5 stages, issued three ways:
//       one lane issuing ten 4 KB row copies | one lane per row (full barrier counts ten arrivals) | four [10 x 256]
//       tensor-map boxes from one lane.
//   k2: three tile sets of 64 threads (K2's plain form); each stage is one [10 x 256] box of X and one of G, and each
//       set writes one [10 x 256] tile of `out` per stage, either with STG.128 from registers (as K2 does) or staged in
//       shared memory and stored with one tensor-map box store (cp.async.bulk.tensor ... bulk_group) from one lane.
//       The ring depth is swept from 64 KB to 200 KB.  `copy` points read only X (1:1 read/write mix).
// Every configuration runs `reps` times after a warm-up; median and spread (max - min) / median are printed.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o stream_mix stream_mix.cu && ./stream_mix
#include <cuda.h>
#include <cuda_runtime.h>
#include <cudaTypedefs.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <vector>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)

constexpr int kRows = 10;
constexpr int kBox = 256;        // tensor-map box width (columns)
constexpr int kMaxStages = 16;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile("{\n.reg .pred P1;\nLAB_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra DONE;\nbra LAB_WAIT;\nDONE:\n}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_row(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void box_load(void* dst, const CUtensorMap* map, int c0, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(0), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void box_store(const CUtensorMap* map, int c0, const void* src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(0), "r"(smem_u32(src)) : "memory");
}
__device__ __forceinline__ float4 lds4(const float* p) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_u32(p)));
    return v;
}
__device__ __forceinline__ void stg4(float* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---- K1: read-only [10 x 1024] stages; 256 consumer threads, one column quad each, as in svgd_pairdist_tma_kernel
enum { kRowsOneLane = 0, kLanePerRow = 1, kFourBoxes = 2 };
constexpr int kK1Cols = 1024;
constexpr int kK1Consumers = kK1Cols / 4;

__global__ void __launch_bounds__(kK1Consumers + 32, 1)
k1_stream(const float* __restrict__ X, const __grid_constant__ CUtensorMap map, int64_t D, int64_t ld, int stages, int mode,
          float* sink) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full_bar[kMaxStages], empty_bar[kMaxStages];
    float* tiles = reinterpret_cast<float*>(smem);
    constexpr int stage_elems = kRows * kK1Cols;
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], mode == kLanePerRow ? kRows : 1);
            mbar_init(&empty_bar[s], kK1Consumers / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int64_t ntiles = D / kK1Cols;   // D is a multiple of the tile width here: every copy is full
    if (tid >= kK1Consumers) {
        const int lane = tid - kK1Consumers;
        const bool issues = mode == kLanePerRow ? lane < kRows : lane == 0;
        if (issues) {
            int it = 0;
            for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
                const int s = it % stages;
                const uint32_t use = it / stages;
                mbar_wait(&empty_bar[s], (use & 1u) ^ 1u);
                float* st = tiles + static_cast<size_t>(s) * stage_elems;
                const int64_t col0 = t * kK1Cols;
                if (mode == kLanePerRow) {
                    mbar_expect(&full_bar[s], kK1Cols * 4u);
                    bulk_row(st + lane * kK1Cols, X + lane * ld + col0, kK1Cols * 4u, &full_bar[s]);
                } else if (mode == kRowsOneLane) {
                    mbar_expect(&full_bar[s], stage_elems * 4u);
                    for (int r = 0; r < kRows; ++r) bulk_row(st + r * kK1Cols, X + r * ld + col0, kK1Cols * 4u, &full_bar[s]);
                } else {
                    mbar_expect(&full_bar[s], stage_elems * 4u);
                    for (int b = 0; b < kK1Cols / kBox; ++b) box_load(st + b * kRows * kBox, &map, static_cast<int>(col0) + b * kBox, &full_bar[s]);
                }
            }
        }
    } else {
        float acc = 0.0f;
        int it = 0;
        // quad layout: [rows][1024] for row copies, [4 boxes][rows][256] for tensor boxes
        const int off = mode == kFourBoxes ? (tid / (kBox / 4)) * kRows * kBox + 4 * (tid % (kBox / 4)) : 4 * tid;
        const int rstride = mode == kFourBoxes ? kBox : kK1Cols;
        for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
            const int s = it % stages;
            const uint32_t use = it / stages;
            mbar_wait(&full_bar[s], use & 1u);
            const float* st = tiles + static_cast<size_t>(s) * stage_elems + off;
#pragma unroll
            for (int r = 0; r < kRows; ++r) {
                const float4 v = lds4(st + r * rstride);
                acc += v.x + v.y + v.z + v.w;
            }
            __syncwarp();
            if ((tid & 31) == 0) mbar_arrive(&empty_bar[s]);
        }
        if (acc == 1234.5f) *sink = acc;
    }
}

// ---- K2 mix: [10 x 256] boxes of X (and G) per stage; three tile sets of 64 threads write one [10 x 256] tile each
enum { kStoreStg = 0, kStoreTma = 1 };
constexpr int kSets = 3;
constexpr int kSetThreads = kBox / 4;
constexpr int kK2Consumers = kSets * kSetThreads;

__global__ void __launch_bounds__(kK2Consumers + 32, 1)
k2_mix(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapG, const __grid_constant__ CUtensorMap mapO,
       float* out, int64_t D, int64_t ld, int nin, int stages, int store) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full_bar[kMaxStages], empty_bar[kMaxStages];
    constexpr int box_elems = kRows * kBox;
    const int stage_elems = nin * box_elems;
    float* tiles = reinterpret_cast<float*>(smem);
    float* staging = tiles + static_cast<size_t>(stages) * stage_elems;   // [kSets][rows][256]
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], kSetThreads / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int64_t ntiles = D / kBox;
    if (tid >= kK2Consumers) {
        if (tid == kK2Consumers) {
            int it = 0;
            for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
                const int s = it % stages;
                const uint32_t use = it / stages;
                mbar_wait(&empty_bar[s], (use & 1u) ^ 1u);
                float* st = tiles + static_cast<size_t>(s) * stage_elems;
                mbar_expect(&full_bar[s], stage_elems * 4u);
                box_load(st, &mapX, static_cast<int>(t * kBox), &full_bar[s]);
                if (nin == 2) box_load(st + box_elems, &mapG, static_cast<int>(t * kBox), &full_bar[s]);
            }
        }
    } else {
        const int set = tid / kSetThreads, q = tid % kSetThreads;
        const bool leader = q == 0;
        float* stg = staging + set * box_elems;
        int it = set;
        for (int64_t t = blockIdx.x + static_cast<int64_t>(set) * gridDim.x; t < ntiles; t += kSets * gridDim.x, it += kSets) {
            const int s = it % stages;
            const uint32_t use = it / stages;
            if (use > 0) mbar_wait(&empty_bar[s], (use - 1u) & 1u);   // previous use was another set's
            mbar_wait(&full_bar[s], use & 1u);
            const float* st = tiles + static_cast<size_t>(s) * stage_elems + 4 * q;
            float4 o[kRows];
#pragma unroll
            for (int r = 0; r < kRows; ++r) {
                o[r] = lds4(st + r * kBox);
                if (nin == 2) {
                    const float4 g = lds4(st + box_elems + r * kBox);
                    o[r].x += g.x; o[r].y += g.y; o[r].z += g.z; o[r].w += g.w;
                }
            }
            __syncwarp();
            if ((tid & 31) == 0) mbar_arrive(&empty_bar[s]);
            const int64_t col0 = t * kBox;
            if (store == kStoreStg) {
#pragma unroll
                for (int r = 0; r < kRows; ++r) stg4(out + r * ld + col0 + 4 * q, o[r]);
            } else {
                // the set's staging buffer is free once the previous box store has read it
                if (leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                asm volatile("bar.sync %0, %1;" ::"r"(1 + set), "n"(kSetThreads) : "memory");
#pragma unroll
                for (int r = 0; r < kRows; ++r) *reinterpret_cast<float4*>(stg + r * kBox + 4 * q) = o[r];
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("bar.sync %0, %1;" ::"r"(1 + set), "n"(kSetThreads) : "memory");
                if (leader) {
                    box_store(&mapO, static_cast<int>(col0), stg);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
        }
        if (store == kStoreTma && leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
}

static PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
    return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
}
static bool encode(CUtensorMap* map, float* M, int64_t D, int64_t ld) {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = encode_fn();
    const cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)kRows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    const cuuint32_t box[2] = {(cuuint32_t)kBox, (cuuint32_t)kRows};
    const cuuint32_t es[2] = {1, 1};
    return fn && fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, M, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct Stats { float med, spread; };
template <class F>
static Stats time_it(F launch, int reps, cudaEvent_t e0, cudaEvent_t e1) {
    std::vector<float> ms;
    launch();   // warm-up
    for (int r = 0; r < reps; ++r) {
        cudaEventRecord(e0);
        launch();
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float v;
        cudaEventElapsedTime(&v, e0, e1);
        ms.push_back(v);
    }
    std::sort(ms.begin(), ms.end());
    return {ms[ms.size() / 2], (ms.back() - ms.front()) / ms[ms.size() / 2]};
}

int main(int argc, char** argv) {
    const int reps = argc > 1 ? atoi(argv[1]) : 9;
    const int64_t D = 100000000, ld = D;   // n = 10, D = 1e8: the flagship shape, 4 GB per matrix
    float *X, *G, *O, *sink;
    CK(cudaMalloc(&X, kRows * ld * 4));
    CK(cudaMalloc(&G, kRows * ld * 4));
    CK(cudaMalloc(&O, kRows * ld * 4));
    CK(cudaMalloc(&sink, 4));
    CK(cudaMemset(X, 0, kRows * ld * 4));
    CK(cudaMemset(G, 0, kRows * ld * 4));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    const int sms = prop.multiProcessorCount;
    printf("{\"device\": \"%s\", \"sms\": %d, \"rows\": %d, \"D\": %lld, \"reps\": %d}\n", prop.name, sms, kRows, (long long)D, reps);
    CUtensorMap mX{}, mG{}, mO{};
    if (!encode(&mX, X, D, ld) || !encode(&mG, G, D, ld) || !encode(&mO, O, D, ld)) { printf("encode failed\n"); return 1; }
    CK(cudaFuncSetAttribute(k1_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    CK(cudaFuncSetAttribute(k2_mix, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);

    // plain device copy of one [10, D] matrix: the "copy bandwidth" reference
    {
        const Stats st = time_it([&] { cudaMemcpyAsync(O, X, kRows * ld * 4, cudaMemcpyDeviceToDevice); }, reps, e0, e1);
        const double bytes = 2.0 * kRows * D * 4;
        printf("{\"bench\": \"memcpy_d2d\", \"read_write\": \"1:1\", \"ms\": %.4f, \"spread\": %.4f, \"TBps\": %.3f}\n", st.med, st.spread, bytes / st.med / 1e9);
        fflush(stdout);
    }
    CK(cudaGetLastError());

    const char* k1_names[] = {"rows_one_lane", "lane_per_row", "four_boxes"};
    for (int stages = 2; stages <= 5; ++stages) {
        for (int mode = 0; mode < 3; ++mode) {
            const int smem = stages * kRows * kK1Cols * 4;
            const Stats st = time_it([&] { k1_stream<<<sms, kK1Consumers + 32, smem>>>(X, mX, D, ld, stages, mode, sink); }, reps, e0, e1);
            CK(cudaGetLastError());
            const double bytes = (double)(D / kK1Cols) * kK1Cols * kRows * 4;
            printf("{\"bench\": \"k1\", \"issue\": \"%s\", \"stages\": %d, \"ring_kb\": %d, \"ms\": %.4f, \"spread\": %.4f, \"TBps\": %.3f}\n",
                   k1_names[mode], stages, smem / 1024, st.med, st.spread, bytes / st.med / 1e9);
            fflush(stdout);
        }
    }
    CK(cudaDeviceSynchronize());

    const char* st_names[] = {"stg128", "tma_box_store"};
    for (int nin = 2; nin >= 1; --nin) {
        for (int ring_kb : {64, 80, 100, 128, 160, 200}) {
            const int stage_bytes = nin * kRows * kBox * 4;
            int stages = ring_kb * 1024 / stage_bytes;
            if (stages > kMaxStages) stages = kMaxStages;
            if (stages < kSets + 1) stages = kSets + 1;   // every set holds a stage while it computes
            for (int store = 0; store < 2; ++store) {
                const int smem = stages * stage_bytes + (store == kStoreTma ? kSets * kRows * kBox * 4 : 0);
                if (smem > 220 * 1024) continue;
                const Stats st = time_it([&] { k2_mix<<<sms, kK2Consumers + 32, smem>>>(mX, mG, mO, O, D, ld, nin, stages, store); }, reps, e0, e1);
                CK(cudaGetLastError());
                const double bytes = (double)(nin + 1) * kRows * D * 4;
                printf("{\"bench\": \"%s\", \"read_write\": \"%d:1\", \"store\": \"%s\", \"stages\": %d, \"ring_kb\": %d, \"ms\": %.4f, \"spread\": %.4f, \"TBps\": %.3f}\n",
                       nin == 2 ? "k2_mix" : "copy", nin, st_names[store], stages, stages * stage_bytes / 1024, st.med, st.spread, bytes / st.med / 1e9);
                fflush(stdout);
            }
        }
    }
    CK(cudaDeviceSynchronize());
    return 0;
}
