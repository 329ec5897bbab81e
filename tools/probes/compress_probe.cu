// compress_probe.cu -- does compute data compression (cuMemCreate with CU_MEM_ALLOCATION_COMP_GENERIC) make the witness
// store stream cheaper?  Two 32 GiB buffers, one plain and one compressible, written with the store shape of k_expand_round
// (256 threads, 2 CTAs/SM through an 85 KiB shared-memory cap, one 256-bit store per 32-byte entry, 8192-entry tiles) and three
// contents: (a) (pseudo-random bit, 0, 0, 0) = the KeccakfRound tiles, (b) four full-entropy words = the worst case (VAL
// entries), (c) zeros.  Then a k_digest-style read-back of each and a 1 GiB D2H copy; digests and copies must agree.
// nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o compress_probe compress_probe.cu -lcuda ; ./compress_probe
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#define DRV(x) do { CUresult r_ = (x); if (r_ != CUDA_SUCCESS) { const char *s_ = nullptr; cuGetErrorString(r_, &s_); printf("%s: %s\n", #x, s_ ? s_ : "?"); exit(1); } } while (0)
#define RT(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e_)); exit(1); } } while (0)

__device__ __forceinline__ uint64_t mix(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL; x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL; x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL; return x ^ (x >> 31);
}
__device__ __forceinline__ void st256(uint64_t *p, uint64_t a, uint64_t b, uint64_t c, uint64_t d) {
    asm volatile("st.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d));
}
// MODE 0: (bit, 0, 0, 0); 1: four full-entropy words; 2: zeros.  One CTA per tile of `tile` entries, as k_expand_round.
template <int T, int MODE>
__global__ void __launch_bounds__(T) k_store(uint64_t *w, uint32_t tile, uint64_t seed) {
    const uint64_t e0 = (uint64_t)blockIdx.x * tile;
    uint64_t *W = w + e0 * 4;
#pragma unroll 8
    for (uint32_t k = threadIdx.x; k < tile; k += T) {
        const uint64_t h = mix(seed ^ (e0 + k));
        if (MODE == 0) st256(W + 4ull * k, h & 1ull, 0, 0, 0);
        else if (MODE == 1) {           // one hash per entry, as in (a): three more hashes per entry make the kernel ALU-bound
            const uint64_t m = h * 0xD6E8FEB86659FD93ULL;
            st256(W + 4ull * k, h, m, m ^ (h >> 29) ^ (h << 35), (m >> 31) + (h << 17));
        }
        else st256(W + 4ull * k, 0, 0, 0, 0);
    }
}
// the read pattern and mixing of k_digest (kernels.cuh)
__global__ void __launch_bounds__(256) k_digest(const uint64_t *wit, uint64_t n, unsigned long long *out) {
    uint64_t acc = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const ulonglong4 v = *reinterpret_cast<const ulonglong4 *>(wit + 4 * i);
        uint64_t h = (i + 1) * 0x9E3779B97F4A7C15ULL;
        h ^= v.x * 0xBF58476D1CE4E5B9ULL + v.y * 0x94D049BB133111EBULL + v.z * 0xD6E8FEB86659FD93ULL + v.w * 0xA0761D6478BD642FULL;
        h ^= h >> 29; h *= 0xBF58476D1CE4E5B9ULL; h ^= h >> 32;
        acc += h;
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    __shared__ uint64_t part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) { uint64_t s = 0; for (int q = 0; q < 8; q++) s += part[q]; atomicAdd(out, (unsigned long long)s); }
}

struct Buf { uint64_t *p; size_t bytes; CUmemGenericAllocationHandle h; int granted; };
static Buf vmm_alloc(CUdevice dev, size_t want, unsigned char comp) {
    CUmemAllocationProp prop{}; prop.type = CU_MEM_ALLOCATION_TYPE_PINNED; prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE; prop.location.id = (int)dev;
    prop.allocFlags.compressionType = comp;
    size_t gran = 0; DRV(cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED));
    Buf b{}; b.bytes = (want + gran - 1) / gran * gran;
    DRV(cuMemCreate(&b.h, b.bytes, &prop, 0));
    CUmemAllocationProp got{}; DRV(cuMemGetAllocationPropertiesFromHandle(&got, b.h)); b.granted = got.allocFlags.compressionType;
    CUdeviceptr va = 0; DRV(cuMemAddressReserve(&va, b.bytes, gran, 0, 0));
    DRV(cuMemMap(va, b.bytes, 0, b.h, 0));
    CUmemAccessDesc ad{}; ad.location = prop.location; ad.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    DRV(cuMemSetAccess(va, b.bytes, &ad, 1));
    b.p = (uint64_t *)va;
    printf("alloc %s: requested comp=%d granted comp=%d, %zu bytes (granularity %zu)\n", comp ? "compressible" : "plain", comp, b.granted, b.bytes, gran);
    return b;
}
static void vmm_free(Buf &b) { DRV(cuMemUnmap((CUdeviceptr)b.p, b.bytes)); DRV(cuMemAddressFree((CUdeviceptr)b.p, b.bytes)); DRV(cuMemRelease(b.h)); }

template <class F> static float timeit(F f, int reps) {
    cudaEvent_t a, b; RT(cudaEventCreate(&a)); RT(cudaEventCreate(&b));
    f(); RT(cudaDeviceSynchronize());
    RT(cudaEventRecord(a)); for (int i = 0; i < reps; i++) f(); RT(cudaEventRecord(b)); RT(cudaEventSynchronize(b));
    RT(cudaGetLastError());
    float ms; RT(cudaEventElapsedTime(&ms, a, b)); cudaEventDestroy(a); cudaEventDestroy(b); return ms / reps;
}

static const uint32_t TILE = 8192;
static void store(uint64_t *w, size_t bytes, int mode, int smem, uint64_t seed) {
    const uint32_t nt = (uint32_t)(bytes / 32 / TILE);
    if (mode == 0) k_store<256, 0><<<nt, 256, smem>>>(w, TILE, seed);
    else if (mode == 1) k_store<256, 1><<<nt, 256, smem>>>(w, TILE, seed);
    else k_store<256, 2><<<nt, 256, smem>>>(w, TILE, seed);
}

int main() {
    DRV(cuInit(0)); RT(cudaSetDevice(0)); RT(cudaFree(0));
    CUdevice dev; DRV(cuDeviceGet(&dev, 0));
    char name[256]; DRV(cuDeviceGetName(name, sizeof name, dev));
    int supported = 0; DRV(cuDeviceGetAttribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev));
    int drv = 0; cuDriverGetVersion(&drv);
    printf("device %s, driver API %d, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = %d\n", name, drv, supported);
    const size_t BYTES = 32ull << 30;
    Buf B[2] = {vmm_alloc(dev, BYTES, CU_MEM_ALLOCATION_COMP_NONE), vmm_alloc(dev, BYTES, supported ? CU_MEM_ALLOCATION_COMP_GENERIC : CU_MEM_ALLOCATION_COMP_NONE)};
    size_t fr = 0, tot = 0; RT(cudaMemGetInfo(&fr, &tot)); printf("cudaMemGetInfo after both allocations: free %.2f GB of %.2f GB\n", fr / 1e9, tot / 1e9);
    const char *arm[2] = {"plain", "compressible"};
    const char *content[3] = {"(a) (bit,0,0,0)", "(b) 4 full-entropy words", "(c) zeros"};
    const int SMEM = 85 * 1024;
    RT(cudaFuncSetAttribute(k_store<256, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    RT(cudaFuncSetAttribute(k_store<256, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    RT(cudaFuncSetAttribute(k_store<256, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    unsigned long long *d_dig; RT(cudaMalloc(&d_dig, 8));
    const size_t CP = 1ull << 30; void *host[2]; RT(cudaMallocHost(&host[0], CP)); RT(cudaMallocHost(&host[1], CP));
    bool all_ok = true;
    for (int mode = 0; mode < 3; mode++) {
        float st[2][3] = {};
        for (int rep = 0; rep < 3; rep++)          // alternated: plain, compressible, plain, ...
            for (int b = 0; b < 2; b++) st[b][rep] = timeit([&] { store(B[b].p, BYTES, mode, SMEM, 12345); }, 10);
        unsigned long long dig[2]; float rd[2], cp[2];
        for (int b = 0; b < 2; b++) {
            store(B[b].p, BYTES, mode, SMEM, 12345); RT(cudaDeviceSynchronize());
            RT(cudaMemset(d_dig, 0, 8)); k_digest<<<1184, 256>>>(B[b].p, BYTES / 32, d_dig); RT(cudaMemcpy(&dig[b], d_dig, 8, cudaMemcpyDeviceToHost));
            rd[b] = timeit([&] { k_digest<<<1184, 256>>>(B[b].p, BYTES / 32, d_dig); }, 10);
            cp[b] = timeit([&] { RT(cudaMemcpyAsync(host[b], (const char *)B[b].p + BYTES / 2, CP, cudaMemcpyDeviceToHost)); }, 3);
        }
        const bool same = dig[0] == dig[1] && memcmp(host[0], host[1], CP) == 0;
        all_ok = all_ok && same;
        for (int b = 0; b < 2; b++) {
            float best = st[b][0]; for (float v : st[b]) best = v < best ? v : best;
            printf("%-26s %-12s store %7.3f ms = %7.1f GB/s (reps %.3f %.3f %.3f)  digest-read %7.3f ms = %7.1f GB/s  D2H 1 GiB %6.2f GB/s\n",
                   content[mode], arm[b], best, BYTES / (best * 1e-3) / 1e9, st[b][0], st[b][1], st[b][2], rd[b], BYTES / (rd[b] * 1e-3) / 1e9, CP / (cp[b] * 1e-3) / 1e9);
        }
        float bp = st[0][0], bc = st[1][0]; for (int r = 0; r < 3; r++) { bp = st[0][r] < bp ? st[0][r] : bp; bc = st[1][r] < bc ? st[1][r] : bc; }
        printf("%-26s compressible/plain store time %.4f  digests %016llx %016llx  same bytes: %s\n", content[mode], bc / bp, dig[0], dig[1], same ? "yes" : "NO");
        fflush(stdout);
    }
    // CTAs per SM on the compressible buffer, content (a): the 85 KiB cap (2) was chosen for uncompressed DRAM row locality
    for (int b = 0; b < 2; b++)
        for (int kb : {120, 85, 70, 50, 0}) {
            if (kb) { RT(cudaFuncSetAttribute(k_store<256, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kb * 1024)); }
            const float ms = timeit([&] { store(B[b].p, BYTES, 0, kb * 1024, 777); }, 10);
            printf("(a) %-12s smem cap %3d KiB (%s CTAs/SM) store %7.3f ms = %7.1f GB/s\n", arm[b], kb, kb == 120 ? "1" : kb == 85 ? "2" : kb == 70 ? "3" : kb == 50 ? "4" : "8", ms, BYTES / (ms * 1e-3) / 1e9);
        }
    for (int b = 0; b < 2; b++) { const float ms = timeit([&] { RT(cudaMemsetAsync(B[b].p, 0, BYTES)); }, 3); printf("cudaMemsetAsync %-12s %7.3f ms = %7.1f GB/s\n", arm[b], ms, BYTES / (ms * 1e-3) / 1e9); }
    cudaFreeHost(host[0]); cudaFreeHost(host[1]); cudaFree(d_dig);
    vmm_free(B[0]); vmm_free(B[1]);
    printf("%s\n", all_ok ? "probe ok: both buffers read back the same bytes" : "probe FAILED: read-back differs");
    return all_ok ? 0 : 1;
}
