// Training-batch pixel sampler: the region-budgeted draw of sample_rays (audio_exp_nerf.py:141-187, data.HeadDataset.sample_pixels) and
// the batch built from it, on the device and graph-capturable.  The contract (keys, regions, selection, order) is written down in
// include/inerf_b200.h above InerfPixelSampleArgs; oracle/pixel_sampler_ref.py restates it in numpy.
//
// Per region the work is an exact top-k of (key << 32 | p) over the region's members:
//   1. hist:    one thread per pixel classifies it, computes its Philox block and counts the high 12 key bits per region (global RED);
//   2. bound:   one CTA per region scans its histogram for the bin where the running count reaches k;
//   3. compact: one thread per pixel again (recomputing Philox is cheaper than storing keys) appends (key << 32 | p) of every member at or
//               below that bin to the region's candidate buffer (warp-aggregated atomics): < k + one bin of candidates;
//   4. select:  one CTA per region bitonic-sorts its candidates in shared memory, keeps the first k and writes, for the rows inside the
//               band, the packed ray, the target, bc_rgb and optionally the coordinates.
#include "common.cuh"
#include "philox.cuh"
#include "rays_parts.cuh"

using namespace inerf;

namespace {

constexpr int kRegions = 4;                                 // rect, norect, mouth, torso (the output order)
constexpr int kBinShift = 20;                               // 4096 bins of the top 12 key bits
constexpr int kBins = 1 << (32 - kBinShift);
constexpr int kCandCap = 2 * INERF_PIXEL_SAMPLER_MAX_K;     // sorted in shared memory: 64 KB of uint64
constexpr int kSelectThreads = 1024;

struct Workspace {
    uint32_t* hist;           // (4, kBins)
    uint32_t* count;          // (4) candidates appended
    int32_t* bound;           // (4) last candidate bin, -1 when k == 0
    unsigned long long* cand; // (4, kCandCap)
};

constexpr size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
constexpr size_t kHistBytes = (size_t)kRegions * kBins * 4 + 256;       // hist, then count (zeroed together) and bound
constexpr size_t kWorkspaceBytes = align256(kHistBytes) + (size_t)kRegions * kCandCap * 8;

Workspace carve(void* base) {
    char* b = static_cast<char*>(base);
    Workspace w;
    w.hist = reinterpret_cast<uint32_t*>(b);
    w.count = reinterpret_cast<uint32_t*>(b + (size_t)kRegions * kBins * 4);
    w.bound = reinterpret_cast<int32_t*>(b + (size_t)kRegions * kBins * 4 + 128);
    w.cand = reinterpret_cast<unsigned long long*>(b + align256(kHistBytes));
    return w;
}

// Frame index read from device memory; -1 when outside [0, F) (then no kernel reads the tables or writes an output).
__device__ __forceinline__ long long frame_of(const InerfPixelSampleArgs& a) {
    const long long f = *reinterpret_cast<const long long*>(a.frame_index);
    return (f >= 0 && f < a.n_frames) ? f : -1;
}

// Region keys of pixel p: key[r] valid when bit r of the returned mask is set.
__device__ __forceinline__ unsigned classify(const InerfPixelSampleArgs& a, long long f, int p, uint32_t (&key)[kRegions]) {
    const int row = p / a.W, col = p - row * a.W;
    const int* b = a.bounds + f * 8;
    const bool rect = row >= b[0] && row <= b[1] && col >= b[2] && col <= b[3];
    const bool mouth = row >= b[4] && row <= b[5] && col >= b[6] && col <= b[7];
    const size_t words = ((size_t)a.H * a.W + 31) >> 5;
    const bool torso = (a.torso_bits[f * words + (p >> 5)] >> (p & 31)) & 1u;
    const Philox4 q = philox_at(reinterpret_cast<const unsigned long long*>(a.rng_state), (uint64_t)p, INERF_RNG_STREAM_PIXELS);
    key[0] = q.x; key[1] = q.x; key[2] = q.y; key[3] = q.z;
    return (rect && !mouth ? 1u : 0u) | (!rect ? 2u : 0u) | (mouth ? 4u : 0u) | (torso ? 8u : 0u);
}

__global__ void __launch_bounds__(256) pixel_hist_kernel(const InerfPixelSampleArgs a, Workspace w) {
    const long long f = frame_of(a);
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < 0 || p >= a.H * a.W) return;
    uint32_t key[kRegions];
    const unsigned m = classify(a, f, p, key);
#pragma unroll
    for (int r = 0; r < kRegions; ++r)
        if (((m >> r) & 1u) && a.k[r] > 0) atomicAdd(&w.hist[r * kBins + (key[r] >> kBinShift)], 1u);
}

// bound[r] = the smallest bin at which the running count reaches k (every bin when the region is short of k; -1 when k == 0)
__global__ void __launch_bounds__(1024) pixel_bound_kernel(const InerfPixelSampleArgs a, Workspace w) {
    constexpr int kPer = kBins / 1024;
    __shared__ uint32_t warp_tot[32];
    __shared__ int32_t bound;
    const int r = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const uint32_t k = (uint32_t)a.k[r];
    if (t == 0) bound = k == 0 ? -1 : kBins - 1;
    uint32_t c[kPer], sum = 0;
#pragma unroll
    for (int i = 0; i < kPer; ++i) { c[i] = w.hist[r * kBins + t * kPer + i]; sum += c[i]; }
    uint32_t incl = sum;                                    // block-wide inclusive scan of the per-thread sums
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        uint32_t v = warp_tot[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += u;
        }
        warp_tot[lane] = v;
    }
    __syncthreads();
    uint32_t run = incl - sum + (warp > 0 ? warp_tot[warp - 1] : 0u);
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
        if (k > 0 && run < k && run + c[i] >= k) bound = t * kPer + i;     // exactly one bin crosses when the region has k members
        run += c[i];
    }
    __syncthreads();
    if (t == 0) w.bound[r] = bound;
}

__global__ void __launch_bounds__(256) pixel_compact_kernel(const InerfPixelSampleArgs a, Workspace w) {
    const long long f = frame_of(a);
    if (f < 0) return;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = p < a.H * a.W;
    uint32_t key[kRegions] = {0u, 0u, 0u, 0u};
    const unsigned m = live ? classify(a, f, p, key) : 0u;
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int r = 0; r < kRegions; ++r) {
        const bool take = ((m >> r) & 1u) && (int)(key[r] >> kBinShift) <= w.bound[r];
        const unsigned ballot = __ballot_sync(0xffffffffu, take);
        if (!ballot) continue;
        const int leader = __ffs(ballot) - 1;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(&w.count[r], (uint32_t)__popc(ballot));
        base = __shfl_sync(0xffffffffu, base, leader);
        const uint32_t slot = base + __popc(ballot & ((1u << lane) - 1u));
        if (take && slot < (uint32_t)kCandCap) w.cand[(size_t)r * kCandCap + slot] = ((unsigned long long)key[r] << 32) | (unsigned)p;
    }
}

__global__ void __launch_bounds__(kSelectThreads) pixel_select_kernel(const InerfPixelSampleArgs a, Workspace w) {
    extern __shared__ unsigned long long s[];
    const int r = blockIdx.x, t = threadIdx.x;
    const int k = a.k[r];
    const long long f = frame_of(a);
    if (k == 0 || f < 0) return;
    const int n = (int)min(w.count[r], (uint32_t)kCandCap);
    int n2 = 1;
    while (n2 < n) n2 <<= 1;
    for (int i = t; i < n2; i += kSelectThreads) s[i] = i < n ? w.cand[(size_t)r * kCandCap + i] : ~0ull;
    __syncthreads();
    for (int size = 2; size <= n2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int q = t; q < (n2 >> 1); q += kSelectThreads) {
                const int i = 2 * q - (q & (stride - 1)), j = i + stride;
                const unsigned long long x = s[i], y = s[j];
                if ((x > y) == ((i & size) == 0)) { s[i] = y; s[j] = x; }
            }
            __syncthreads();
        }
    }
    int row0 = 0;
    for (int i = 0; i < r; ++i) row0 += a.k[i];
    const int m = min(k, n);                                // n < k only for a region short of members: its tail rows are not written
    const float* c2w = a.poses + f * 12;
    const size_t hw = (size_t)a.H * a.W;
    for (int i = t; i < m; i += kSelectThreads) {
        const int o = row0 + i - a.first;
        if (o < 0 || o >= a.count) continue;
        const int p = (int)(unsigned)(s[i] & 0xffffffffull);
        const int row = p / a.W, col = p - row * a.W;
        float d[3];
        pixel_dir((float)row, (float)col, a.focal, a.cx, a.cy, c2w, 4, d);
        store_ray(a.rays + (size_t)o * 11, c2w[3], c2w[7], c2w[11], d[0], d[1], d[2], a.near_, a.far_);
        const uint8_t* px = a.frames + ((size_t)f * hw + p) * 3;
        const float* bc = a.bc_img + (size_t)p * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            // torch divides a CUDA tensor by a host scalar as a product with the rounded reciprocal: HeadDataset's target_s bits
            a.target[(size_t)o * 3 + c] = __fmul_rn((float)px[c], 1.0f / 255.0f);
            a.bc_rgb[(size_t)o * 3 + c] = bc[c];
        }
        if (a.coords) {
            a.coords[(size_t)o * 2] = row;
            a.coords[(size_t)o * 2 + 1] = col;
        }
    }
}

int check_shapes(const InerfPixelSampleArgs* a, const char* what) {
    if (a->H <= 0 || a->W <= 0 || (int64_t)a->H * a->W > INERF_PIXEL_SAMPLER_MAX_PIXELS || a->n_frames <= 0) {
        set_error("%s: bad H / W / n_frames (H * W <= %d pixels)", what, INERF_PIXEL_SAMPLER_MAX_PIXELS);
        return INERF_E_SHAPE;
    }
    int64_t n_rand = 0;
    for (int r = 0; r < kRegions; ++r) {
        if (a->k[r] < 0) {
            set_error("%s: negative region budget", what);
            return INERF_E_SHAPE;
        }
        if (a->k[r] > INERF_PIXEL_SAMPLER_MAX_K) {
            set_error("%s: region budget %d above the %d rows one CTA sorts", what, a->k[r], INERF_PIXEL_SAMPLER_MAX_K);
            return INERF_E_UNSUPPORTED;
        }
        n_rand += a->k[r];
    }
    if (a->first < 0 || a->count < 0 || (int64_t)a->first + a->count > n_rand) {
        set_error("%s: band [first, first + count) outside the N_rand rows", what);
        return INERF_E_SHAPE;
    }
    return INERF_OK;
}

}  // namespace

extern "C" int inerf_pixel_sampler_workspace_bytes(const InerfPixelSampleArgs* args, size_t* bytes) {
    if (!args || !bytes) return fail(INERF_E_ARG, "inerf_pixel_sampler_workspace_bytes: NULL pointer");
    if (int rc = check_shapes(args, "inerf_pixel_sampler_workspace_bytes")) return rc;
    *bytes = kWorkspaceBytes;
    return INERF_OK;
}

extern "C" int inerf_sample_train_pixels(const InerfPixelSampleArgs* args, void* workspace, size_t workspace_bytes, void* stream) {
    if (!args) return fail(INERF_E_ARG, "inerf_sample_train_pixels: args is NULL");
    const InerfPixelSampleArgs& a = *args;
    if (int rc = check_shapes(args, "inerf_sample_train_pixels")) return rc;
    if (!workspace || !a.frame_index || !a.bounds || !a.torso_bits || !a.poses || !a.frames || !a.bc_img || !a.rng_state || !a.rays ||
        !a.target || !a.bc_rgb)
        return fail(INERF_E_ARG, "inerf_sample_train_pixels: NULL pointer");
    if (workspace_bytes < kWorkspaceBytes || ((uintptr_t)workspace & 255))
        return fail(INERF_E_SHAPE, "inerf_sample_train_pixels: workspace smaller than inerf_pixel_sampler_workspace_bytes or not 256-byte aligned");
    if (a.count == 0) return INERF_OK;
    static_assert(kCandCap * 8 <= 227 * 1024, "candidate sort exceeds shared memory");
    static thread_local int configured_dev = -1;
    int dev = 0;
    cudaGetDevice(&dev);
    if (configured_dev != dev) {
        cudaError_t e = cudaFuncSetAttribute(pixel_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCandCap * 8);
        if (e != cudaSuccess) {
            set_error("inerf_sample_train_pixels: setup: %s", cudaGetErrorString(e));
            return (int)e;
        }
        configured_dev = dev;
    }
    cudaStream_t s = as_stream(stream);
    const Workspace w = carve(workspace);
    const int hw = a.H * a.W, blocks = (hw + 255) / 256;
    cudaError_t e = cudaMemsetAsync(workspace, 0, kHistBytes, s);
    if (e != cudaSuccess) {
        set_error("inerf_sample_train_pixels: %s", cudaGetErrorString(e));
        return (int)e;
    }
    pixel_hist_kernel<<<blocks, 256, 0, s>>>(a, w);
    pixel_bound_kernel<<<kRegions, 1024, 0, s>>>(a, w);
    pixel_compact_kernel<<<blocks, 256, 0, s>>>(a, w);
    pixel_select_kernel<<<kRegions, kSelectThreads, kCandCap * 8, s>>>(a, w);
    return check_launch("inerf_sample_train_pixels");
}
