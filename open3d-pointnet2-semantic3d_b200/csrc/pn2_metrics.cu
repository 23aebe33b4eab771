// pn2_metrics.cu -- evaluation on the device: arg-max + confusion-matrix update in one pass
// (util/metric.py:7-83 fed by train.py:246-251 / predict.py:90, which copy the logits to the host, take
// np.argmax and count with a Python double loop).
//
// Each block counts into its own C x C histogram of 32-bit counters in shared memory and adds only the non-zero
// bins to the caller's uint64 matrix at the end.  The bins are few and hot (the 9-class head: 81 bins, most points
// of a batch in a handful of them), so lanes of a warp that hit the same bin are combined before the shared atomic
// (__match_any_sync), and the grid stays at a few blocks per SM: every block costs up to C*C global atomics onto
// the same C*C addresses, which the L2 atomic units serialise (NOTES.md, the 9-class head's wgrad).
#include "pn2_common.cuh"

namespace pn2 {
namespace {

constexpr int kMetricThreads = 256;
constexpr int kMetricWarps = kMetricThreads / 32;
constexpr int kMetricMaxClasses = 128;  // 128 x 128 x 4 B = 64 KB of histogram
constexpr int kNoBin = -2;               // a lane without a row in this tile
constexpr int kSkipBin = -1;             // a row or pair whose label lies outside [0, C)

__device__ __forceinline__ void zero_histogram(unsigned *hist, int bins, unsigned *skipped) {
    for (int i = threadIdx.x; i < bins; i += blockDim.x) hist[i] = 0u;
    if (threadIdx.x == 0) *skipped = 0u;
    __syncthreads();
}

// Every lane of the warp calls this with its bin (kNoBin: nothing to count).
__device__ __forceinline__ void count_bin(int bin, unsigned *hist, unsigned *skipped) {
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin != kNoBin && (int)(threadIdx.x & 31) == __ffs(peers) - 1) {
        if (bin >= 0) atomicAdd(&hist[bin], (unsigned)__popc(peers));
        else atomicAdd(skipped, (unsigned)__popc(peers));
    }
}

__device__ __forceinline__ void flush_histogram(const unsigned *hist, int bins, const unsigned *skipped,
                                                unsigned long long *cm, unsigned long long *skipped_out) {
    __syncthreads();
    for (int i = threadIdx.x; i < bins; i += blockDim.x) {
        const unsigned v = hist[i];
        if (v) atomicAdd(cm + i, (unsigned long long)v);
    }
    if (threadIdx.x == 0 && *skipped) atomicAdd(skipped_out, (unsigned long long)*skipped);
}

// np.argmax: the first maximum; a NaN beats every number and the first NaN wins (a row of -inf gives 0).
// Written with explicit isnan, since fmaxf would drop the NaN.
__device__ __forceinline__ int argmax_row(const float *x, int C) {
    float best = x[0];
    int pd = 0;
    for (int c = 1; c < C && !isnan(best); ++c) {
        const float v = x[c];
        if (v > best || isnan(v)) {
            best = v;
            pd = c;
        }
    }
    return pd;
}

// One warp per tile of 32 rows, one lane per row.  A row is only C*4 bytes and, for C = 9, not 16-byte aligned,
// so the warp first stages the tile's contiguous 32*C floats into shared memory with coalesced (float4 when the
// logits are 16-byte aligned: every tile starts at a multiple of 128*C bytes) loads, at a row pitch S = C | 1 so
// that the lanes' row reads hit distinct banks; then every lane scans its own row there.
__global__ void __launch_bounds__(kMetricThreads) confusion_logits_kernel(
    long rows, int C, int S, const float *__restrict__ logits, const int *__restrict__ labels,
    unsigned long long *__restrict__ cm, unsigned long long *__restrict__ skipped, int *__restrict__ pred_out) {
    extern __shared__ unsigned smem_u[];
    const int bins = C * C, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned *hist = smem_u, *nskip = smem_u + bins;
    float *stage = reinterpret_cast<float *>(smem_u + bins + 1) + warp * 32 * S;
    zero_histogram(hist, bins, nskip);
    pdl_enter();
    const bool vec = (reinterpret_cast<uintptr_t>(logits) & 15) == 0;
    const long tiles = ceil_div<long>(rows, 32);
    for (long t = (long)blockIdx.x * kMetricWarps + warp; t < tiles; t += (long)gridDim.x * kMetricWarps) {
        const long r0 = t * 32;
        const int nr = (int)min(32L, rows - r0), n = nr * C;
        const float *src = logits + r0 * C;
        const int gt = lane < nr ? __ldg(labels + r0 + lane) : -1;  // in flight while the tile is staged
        int e = lane;
        if (vec) {
            const int n4 = n >> 2;
            for (int q = lane; q < n4; q += 32) {
                const float4 v = __ldg(reinterpret_cast<const float4 *>(src) + q);
                int r = (4 * q) / C, c = 4 * q - r * C;
                const float vs[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    stage[r * S + c] = vs[j];
                    if (++c == C) c = 0, ++r;
                }
            }
            e = 4 * n4 + lane;
        }
        for (; e < n; e += 32) {
            const int r = e / C;
            stage[r * S + e - r * C] = __ldg(src + e);
        }
        __syncwarp();
        int bin = kNoBin;
        if (lane < nr) {
            const long row = r0 + lane;
            const int pd = argmax_row(stage + lane * S, C);
            if (pred_out) pred_out[row] = pd;
            bin = gt >= 0 && gt < C ? gt * C + pd : kSkipBin;
        }
        count_bin(bin, hist, nskip);
        __syncwarp();  // the next tile overwrites this warp's staging rows
    }
    flush_histogram(hist, bins, nskip, cm, skipped);
}

// Label pairs (sklearn's confusion_matrix(labels=range(C)): a pair with gt or pd outside [0, C) is dropped).
__global__ void __launch_bounds__(kMetricThreads) confusion_labels_kernel(
    long n, int C, const int *__restrict__ gt, const int *__restrict__ pd, unsigned long long *__restrict__ cm,
    unsigned long long *__restrict__ skipped) {
    extern __shared__ unsigned smem_u[];
    const int bins = C * C;
    unsigned *hist = smem_u, *nskip = smem_u + bins;
    zero_histogram(hist, bins, nskip);
    pdl_enter();
    // the loop bound is block-uniform, so every lane of a warp reaches count_bin together
    for (long base = (long)blockIdx.x * blockDim.x; base < n; base += (long)gridDim.x * blockDim.x) {
        const long i = base + threadIdx.x;
        int bin = kNoBin;
        if (i < n) {
            const int g = __ldg(gt + i), p = __ldg(pd + i);
            bin = g >= 0 && g < C && p >= 0 && p < C ? g * C + p : kSkipBin;
        }
        count_bin(bin, hist, nskip);
    }
    flush_histogram(hist, bins, nskip, cm, skipped);
}

// Grid: enough blocks for the work, at most `per_sm` per SM (each block flushes up to C*C global atomics onto the
// same addresses), and never fewer than needed to keep a block's count of rows below 2^31 (32-bit bins).
int metric_grid(long work_items, long items_per_block_pass, int per_sm) {
    long g = ceil_div<long>(work_items, items_per_block_pass);
    g = g < (long)num_sms() * per_sm ? g : (long)num_sms() * per_sm;
    const long floor_blocks = ceil_div<long>(work_items, 1L << 31);
    return (int)(g > floor_blocks ? g : floor_blocks);
}

int metric_blocks_per_sm(size_t smem) { return smem <= 96 * 1024 ? 2 : 1; }

}  // namespace
}  // namespace pn2

using namespace pn2;

PN2_API int pn2_confusion_from_logits(long rows, int C, const float *logits, const int *labels,
                                      unsigned long long *cm, unsigned long long *skipped, int *pred_out,
                                      pn2_stream_t s) {
    PN2_REQUIRE(rows >= 0 && C >= 1);
    if (C > kMetricMaxClasses) return PN2_EUNSUPPORTED;
    if (rows == 0) return PN2_OK;
    PN2_REQUIRE_PTR(logits);
    PN2_REQUIRE_PTR(labels);
    PN2_REQUIRE_PTR(cm);
    PN2_REQUIRE_PTR(skipped);
    const int S = C | 1;
    const size_t smem = sizeof(unsigned) * ((size_t)C * C + 1) + sizeof(float) * kMetricWarps * 32 * S;
    int rc = opt_in_dyn_smem(confusion_logits_kernel, smem);
    if (rc) return rc;
    const int grid = metric_grid(rows, 32L * kMetricWarps, metric_blocks_per_sm(smem));
    launch_k(confusion_logits_kernel, grid, kMetricThreads, smem, as_stream(s), rows, C, S, logits, labels, cm,
             skipped, pred_out);
    return finish_launch();
}

PN2_API int pn2_confusion_from_labels(long n, int C, const int *gt, const int *pd, unsigned long long *cm,
                                      unsigned long long *skipped, pn2_stream_t s) {
    PN2_REQUIRE(n >= 0 && C >= 1);
    if (C > kMetricMaxClasses) return PN2_EUNSUPPORTED;
    if (n == 0) return PN2_OK;
    PN2_REQUIRE_PTR(gt);
    PN2_REQUIRE_PTR(pd);
    PN2_REQUIRE_PTR(cm);
    PN2_REQUIRE_PTR(skipped);
    const size_t smem = sizeof(unsigned) * ((size_t)C * C + 1);
    int rc = opt_in_dyn_smem(confusion_labels_kernel, smem);
    if (rc) return rc;
    const int grid = metric_grid(n, kMetricThreads, metric_blocks_per_sm(smem));
    launch_k(confusion_labels_kernel, grid, kMetricThreads, smem, as_stream(s), n, C, gt, pd, cm, skipped);
    return finish_launch();
}
