// msm_sort.cu — scalar recoding and bucket sort for the MSM (field independent).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include "msm.cuh"

namespace sb {

int g_msm_tuning[12] = {0};

// ------------------------------------------------------------------------------------------------
// digits: thread i recodes scalar i into W signed digits (reference _getChunk extracts unsigned chunks;
// signed recoding halves the bucket count and is free because negating an affine point is free).
// entries are written window-major (keys[w*n + i]) so every store is coalesced.
// ------------------------------------------------------------------------------------------------
__global__ void k_digits(const uint8_t* __restrict__ scalars, uint32_t sbytes, uint64_t n, MsmGeom g,
                         uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w32[17];                       // up to 64-byte scalars + 1 guard word
    const uint8_t* s = scalars + i * sbytes;
    if (sbytes == 32 && ((uintptr_t)scalars & 15) == 0) {
        const uint4* p = reinterpret_cast<const uint4*>(s);
        uint4 a = __ldg(p), b = __ldg(p + 1);
        w32[0] = a.x; w32[1] = a.y; w32[2] = a.z; w32[3] = a.w; w32[4] = b.x; w32[5] = b.y; w32[6] = b.z; w32[7] = b.w;
#pragma unroll
        for (int k = 8; k < 17; k++) w32[k] = 0;
    } else {
#pragma unroll
        for (int k = 0; k < 17; k++) w32[k] = 0;
        for (uint32_t k = 0; k < sbytes; k++) w32[k >> 2] |= (uint32_t)s[k] << (8 * (k & 3));
    }
    const uint32_t cmask = (1u << g.c) - 1, half = 1u << (g.c - 1);
    uint32_t carry = 0;
    for (int w = 0; w < g.W; w++) {
        uint32_t bit = (uint32_t)w * g.c, wi = bit >> 5, sh = bit & 31;
        uint64_t two = (uint64_t)w32[wi] | ((uint64_t)(wi + 1 < 17 ? w32[wi + 1] : 0) << 32);
        uint32_t raw = ((uint32_t)(two >> sh) & cmask) + carry;
        uint32_t key, val = (uint32_t)i;
        if (raw > half) { raw = (1u << g.c) - raw; carry = 1; val |= 0x80000000u; } else carry = 0;
        if (g.precomp) { key = raw ? raw - 1 : MSM_INVALID_KEY; val = (uint32_t)((uint64_t)w * g.stride + g.first + i) | (val & 0x80000000u); }
        else key = raw ? (uint32_t)w * g.B + raw - 1 : MSM_INVALID_KEY;
        keys[(uint64_t)w * n + i] = key;
        vals[(uint64_t)w * n + i] = val;
    }
}

// number of valid (non-zero-digit) entries = first index whose sorted key is INVALID, then the counts derived from it
__global__ void k_count_valid(const uint32_t* __restrict__ keys, uint64_t total, uint64_t* __restrict__ out, uint32_t T, uint32_t seg_lo, uint64_t wave) {
    if (blockIdx.x | threadIdx.x) return;
    uint64_t lo = 0, hi = total;
    while (lo < hi) { uint64_t mid = (lo + hi) >> 1; if (keys[mid] == MSM_INVALID_KEY) hi = mid; else lo = mid + 1; }
    msm_fill_counts(out, lo, T, seg_lo, wave);
}

int msm_sm_count() {
    static int sm_count = 0;
    if (!sm_count) { int dev = 0; cudaGetDevice(&dev); if (cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sm_count <= 0) sm_count = 148; }
    return sm_count;
}

// ---- output positions of a batched-affine round (msm_pair.cuh): exclusive sum of the per-slot output counts
size_t msm_pair_scan_tmp_bytes(uint64_t items) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)items);
    return bytes;
}
int msm_pair_scan(const uint32_t* counts, uint32_t* pos, uint64_t items, void* tmp, size_t tmp_bytes, cudaStream_t stream) {
    cudaError_t e = cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, counts, pos, (int)items, stream);
    return (int)(e != cudaSuccess ? e : cudaGetLastError());
}

int msm_sort_entries(const uint8_t* d_scalars, uint32_t sbytes, uint64_t n, MsmGeom g, MsmScratch& scratch,
                     cudaStream_t stream, MsmSorted* out, MsmLaunchStats* stats) {
    const uint64_t total = n * (uint64_t)g.W;
    const uint64_t nbuckets = (uint64_t)g.windows() * g.B;
    if (sbytes == 0 || sbytes > 64) return (int)cudaErrorInvalidValue;
    int key_bits = 1; while ((1ull << key_bits) < nbuckets) key_bits++;
    int end_bit = key_bits + 1 > 32 ? 32 : key_bits + 1;   // INVALID (all ones) sorts after every valid key
    size_t sort_tmp = 0;
    cub::DoubleBuffer<uint32_t> kb(nullptr, nullptr), vb(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, kb, vb, (uint64_t)total, 0, end_bit, stream);
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t o_keys0 = 0, o_keys1 = o_keys0 + al(total * 4), o_vals0 = o_keys1 + al(total * 4), o_vals1 = o_vals0 + al(total * 4);
    size_t o_tmp = o_vals1 + al(total * 4), o_counts = o_tmp + al(sort_tmp);
    uint8_t* base = (uint8_t*)scratch.get(o_counts + 256);
    if (!base) return (int)cudaErrorMemoryAllocation;
    uint32_t* keys0 = (uint32_t*)(base + o_keys0); uint32_t* keys1 = (uint32_t*)(base + o_keys1);
    uint32_t* vals0 = (uint32_t*)(base + o_vals0); uint32_t* vals1 = (uint32_t*)(base + o_vals1);
    uint64_t* counts = (uint64_t*)(base + o_counts);
    int launches = 0;
    ProfScope prof(stats, PROF_SORT, stream);
    k_digits<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(d_scalars, sbytes, n, g, keys0, vals0); launches++;
    kb = cub::DoubleBuffer<uint32_t>(keys0, keys1); vb = cub::DoubleBuffer<uint32_t>(vals0, vals1);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(base + o_tmp, sort_tmp, kb, vb, (uint64_t)total, 0, end_bit, stream);
    if (e != cudaSuccess) return (int)e;
    launches += 2 + (end_bit + 7) / 8;   // histogram + scan + one onesweep pass per 8 key bits
    // target entries per thread: dense buckets keep the head partials at <= ~2 per bucket; then whole-wave fitting on the device
    uint32_t T = MSM_SEG;
    const bool adaptive = g_msm_tuning[5] >= 0 && g_msm_tuning[7] <= 0;
    if (adaptive) { const uint64_t avg = nbuckets ? total / nbuckets : 0; while (T < 256 && avg > 2ull * T) T <<= 1; }
    if (g_msm_tuning[7] > 0) T = (uint32_t)g_msm_tuning[7];
    const uint64_t wave = adaptive ? (uint64_t)msm_sm_count() * 4 * MSM_ACC_THREADS : 0;     // 4 CTAs of 128 threads per SM (2 for the extension-field kernels: same fit)
    const uint32_t seg_lo = adaptive ? (T == (uint32_t)MSM_SEG ? 16u : T / 2) : T;
    k_count_valid<<<1, 1, 0, stream>>>(kb.Current(), total, counts, T, seg_lo, wave); launches++;
    prof.end();
    out->seg_lo = seg_lo;
    out->keys = kb.Current(); out->vals = vb.Current(); out->counts = counts; out->n = n; out->total = total; out->g = g;
    if (stats) stats->launches += launches;
    return (int)cudaGetLastError();
}

}  // namespace sb
