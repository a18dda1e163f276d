// LOFOutlierErrorDetector: exact one-dimensional local outlier factor over one float64 column.
//
// In one dimension the k nearest neighbours of a value are a window of k + 1 consecutive entries of
// the sorted column, so the detector is one radix sort plus three stencil passes:
//   fill     NULL -> median of the non-NULL values, -0.0 -> +0.0, order-preserving uint64 keys; the
//            NULL rows are sorted last and then merged into the run of median-valued entries by row
//   sort     cub::DeviceRadixSort::SortPairs on (key, row): stable, so ties keep row order
//   kdist    per sorted position: the leftmost window [l, l + k] minimising
//            d(l) = max(s[i] - s[l], s[l + k] - s[i]) (two binary searches), kdist = d(l*)
//   lrd      1 / (sum_j max(|s[i] - s[j]|, kdist[j]) / k + 1e-10)
//   score    lof = (sum_j lrd[j] / lrd[i]) / k;  flagged iff lof > 1.5
// Sums run over the window in ascending sorted position, skipping i, with explicit round-to-nearest
// double operations (no contraction), so the result is bit-identical to the host definition
// (tests/lof_reference.py).  The stencil kernels stage a tile of kLofTile sorted positions plus a
// k-entry halo on each side in shared memory.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace {

constexpr int kLofThreads = 256;
constexpr int kLofTile = 1024;                       // sorted positions per tile
constexpr int kLofPerThread = kLofTile / kLofThreads;
constexpr int kLofCtasPerSm = 4;
constexpr int kLofMaxK = 64;
constexpr int kLofSpan = kLofTile + 2 * kLofMaxK;    // tile + halo
constexpr unsigned long long kNullKey = ~0ull;       // above every non-NaN key: NULLs sort last

struct LofParams {
    double median;
    int64_t n_valid;            // non-NULL values
    int64_t run_lo, run_hi;     // sorted positions of the non-NULL entries equal to the median
    unsigned long long flagged; // flagged rows inside [row_begin, row_begin + row_count)
};

__device__ __forceinline__ unsigned long long lof_key(double v) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(v);
    return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}

__device__ __forceinline__ double lof_value(unsigned long long k) {
    const unsigned long long u = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)u);
}

__global__ void __launch_bounds__(kLofThreads) k_lof_keys(const double* __restrict__ col, int64_t n,
                                                          unsigned long long* __restrict__ keys,
                                                          int32_t* __restrict__ rows) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) {
        const double v = __ldcs(col + r);
        keys[r] = v != v ? kNullKey : lof_key(v == 0.0 ? 0.0 : v);
        rows[r] = (int32_t)r;
    }
}

// First position in [lo, hi) whose key is >= (or > when `upper`) `key`.
__device__ int64_t lof_bound(const unsigned long long* keys, int64_t lo, int64_t hi, unsigned long long key,
                             bool upper) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const unsigned long long k = keys[mid];
        if (upper ? k <= key : k < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// One thread: NULL count, median (np.median: the middle value, or the mean of the two middle values)
// and the run of sorted entries equal to it.
__global__ void k_lof_median(const unsigned long long* __restrict__ keys, int64_t n, LofParams* __restrict__ p) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const int64_t c = lof_bound(keys, 0, n, kNullKey, false);
    p->n_valid = c;
    p->flagged = 0;
    p->median = 0.0;
    p->run_lo = p->run_hi = 0;
    if (c == 0) return;
    const double a = lof_value(keys[(c - 1) >> 1]), b = lof_value(keys[c >> 1]);
    double m = (c & 1) ? a : __ddiv_rn(__dadd_rn(a, b), 2.0);
    if (m == 0.0) m = 0.0;
    const unsigned long long km = lof_key(m);
    p->median = m;
    p->run_lo = lof_bound(keys, 0, c, km, false);
    p->run_hi = lof_bound(keys, p->run_lo, c, km, true);
}

__device__ int64_t lof_rows_below(const int32_t* rows, int64_t len, int32_t row) {
    int64_t lo = 0, hi = len;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (rows[mid] < row) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Sorted keys (NULLs last) -> filled sorted values s and their rows.  The NULL rows take the median and
// are merged, by row, into the run [run_lo, run_hi) of entries equal to it; entries after the run move
// up by the NULL count.
__global__ void __launch_bounds__(kLofThreads) k_lof_place(const unsigned long long* __restrict__ keys,
                                                           const int32_t* __restrict__ rows, int64_t n,
                                                           const LofParams* __restrict__ p, double* __restrict__ s,
                                                           int32_t* __restrict__ perm) {
    const int64_t c = p->n_valid;
    if (c == 0) return;
    const int64_t lo = p->run_lo, hi = p->run_hi, n_null = n - c;
    const double m = p->median;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int32_t row = rows[i];
        int64_t dst;
        double v;
        if (i < lo) {
            dst = i;
            v = lof_value(keys[i]);
        } else if (i < hi) {
            dst = i + lof_rows_below(rows + c, n_null, row);
            v = m;
        } else if (i < c) {
            dst = i + n_null;
            v = lof_value(keys[i]);
        } else {
            dst = lo + (i - c) + lof_rows_below(rows + lo, hi - lo, row);
            v = m;
        }
        s[dst] = v;
        perm[dst] = row;
    }
}

// sh[j] = src[base + j] for the tile starting at sorted position t0 (base = t0 - k), 0 outside [0, n).
__device__ __forceinline__ void lof_load_tile(const double* __restrict__ src, int64_t n, int64_t base, int span,
                                              double* sh) {
    for (int j = threadIdx.x; j < span; j += blockDim.x) {
        const int64_t g = base + j;
        sh[j] = (g >= 0 && g < n) ? src[g] : 0.0;
    }
}

__global__ void __launch_bounds__(kLofThreads) k_lof_kdist(const double* __restrict__ s, int64_t n, int k,
                                                           const LofParams* __restrict__ p,
                                                           double* __restrict__ kdist, uint8_t* __restrict__ off) {
    __shared__ double sh_s[kLofSpan];
    if (p->n_valid == 0) return;
    for (int64_t t0 = (int64_t)blockIdx.x * kLofTile; t0 < n; t0 += (int64_t)gridDim.x * kLofTile) {
        const int64_t base = t0 - k;
        __syncthreads();
        lof_load_tile(s, n, base, kLofTile + 2 * k, sh_s);
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kLofPerThread; ++q) {
            const int64_t i = t0 + q * kLofThreads + threadIdx.x;
            if (i >= n) break;
            auto S = [&](int64_t x) { return sh_s[x - base]; };   // s[x] for x in [i - k, i + k]
            const double si = S(i);
            const int64_t L = i - k > 0 ? i - k : 0;
            const int64_t R = i < n - 1 - k ? i : n - 1 - k;
            // l0: first window whose right reach is at least its left reach (the predicate is monotone:
            // s[i] - s[l] never increases with l, s[l + k] - s[i] never decreases)
            int64_t a = L, b = R + 1;
            while (a < b) {
                const int64_t mid = (a + b) >> 1;
                if (__dsub_rn(S(mid + k), si) >= __dsub_rn(si, S(mid))) b = mid; else a = mid + 1;
            }
            const int64_t l0 = a;
            int64_t ls = l0;
            double d = l0 <= R ? __dsub_rn(S(l0 + k), si) : 0.0;
            if (l0 > L) {
                const double vl = __dsub_rn(si, S(l0 - 1));
                if (l0 > R || vl <= d) {
                    // left of l0, d(l) = s[i] - s[l]: the leftmost window with that same distance
                    int64_t a2 = L, b2 = l0 - 1;
                    while (a2 < b2) {
                        const int64_t mid = (a2 + b2) >> 1;
                        if (__dsub_rn(si, S(mid)) <= vl) b2 = mid; else a2 = mid + 1;
                    }
                    ls = a2;
                    d = vl;
                }
            }
            kdist[i] = d;
            off[i] = (uint8_t)(i - ls);
        }
    }
}

__global__ void __launch_bounds__(kLofThreads) k_lof_lrd(const double* __restrict__ s,
                                                         const double* __restrict__ kdist,
                                                         const uint8_t* __restrict__ off, int64_t n, int k,
                                                         const LofParams* __restrict__ p, double* __restrict__ lrd) {
    __shared__ double sh_s[kLofSpan];
    __shared__ double sh_k[kLofSpan];
    if (p->n_valid == 0) return;
    const double kd = (double)k;
    for (int64_t t0 = (int64_t)blockIdx.x * kLofTile; t0 < n; t0 += (int64_t)gridDim.x * kLofTile) {
        const int64_t base = t0 - k;
        __syncthreads();
        lof_load_tile(s, n, base, kLofTile + 2 * k, sh_s);
        lof_load_tile(kdist, n, base, kLofTile + 2 * k, sh_k);
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kLofPerThread; ++q) {
            const int64_t i = t0 + q * kLofThreads + threadIdx.x;
            if (i >= n) break;
            auto S = [&](int64_t x) { return sh_s[x - base]; };
            auto KD = [&](int64_t x) { return sh_k[x - base]; };
            const double si = S(i);
            const int64_t l = i - off[i];
            double acc = 0.0;
            for (int64_t j = l; j <= l + k; ++j) {
                if (j == i) continue;
                acc = __dadd_rn(acc, fmax(fabs(__dsub_rn(si, S(j))), KD(j)));
            }
            lrd[i] = __ddiv_rn(1.0, __dadd_rn(__ddiv_rn(acc, kd), 1e-10));
        }
    }
}

__global__ void __launch_bounds__(kLofThreads) k_lof_score(const double* __restrict__ lrd,
                                                           const uint8_t* __restrict__ off,
                                                           const int32_t* __restrict__ perm, int64_t n, int k,
                                                           int64_t row_begin, int64_t row_count,
                                                           LofParams* __restrict__ p, uint32_t* __restrict__ bitmap,
                                                           double* __restrict__ out_lof) {
    __shared__ double sh_l[kLofSpan];
    if (p->n_valid == 0) return;
    unsigned int mine = 0;
    for (int64_t t0 = (int64_t)blockIdx.x * kLofTile; t0 < n; t0 += (int64_t)gridDim.x * kLofTile) {
        const int64_t base = t0 - k;
        __syncthreads();
        lof_load_tile(lrd, n, base, kLofTile + 2 * k, sh_l);
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kLofPerThread; ++q) {
            const int64_t i = t0 + q * kLofThreads + threadIdx.x;
            if (i >= n) break;
            auto LR = [&](int64_t x) { return sh_l[x - base]; };
            const double li = LR(i);
            const int64_t l = i - off[i];
            double acc = 0.0;
            for (int64_t j = l; j <= l + k; ++j) {
                if (j == i) continue;
                acc = __dadd_rn(acc, __ddiv_rn(LR(j), li));
            }
            const double lof = __ddiv_rn(acc, (double)k);
            const int64_t row = perm[i];
            if (out_lof) out_lof[row] = lof;
            const int64_t rel = row - row_begin;
            if (lof > 1.5 && rel >= 0 && rel < row_count) {
                atomicOr(bitmap + (rel >> 5), 1u << (rel & 31));
                ++mine;
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&p->flagged, (unsigned long long)mine);
}

// Workspace carve-up (256-byte aligned pieces).
struct LofLayout {
    size_t keys[2], rows[2], kdist, lrd, off, params, temp, temp_bytes, total;
};

size_t lof_align(size_t x) { return (x + 255) & ~(size_t)255; }

cudaError_t lof_layout(int64_t n, LofLayout* out) {
    size_t temp_bytes = 0;
    cub::DoubleBuffer<unsigned long long> dk(nullptr, nullptr);
    cub::DoubleBuffer<int32_t> dv(nullptr, nullptr);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, dk, dv, (int)n, 0, 64);
    if (e != cudaSuccess) return e;
    size_t at = 0;
    auto take = [&](size_t bytes) { const size_t here = at; at += lof_align(bytes); return here; };
    out->keys[0] = take((size_t)n * 8);
    out->keys[1] = take((size_t)n * 8);
    out->rows[0] = take((size_t)n * 4);
    out->rows[1] = take((size_t)n * 4);
    out->kdist = take((size_t)n * 8);
    out->lrd = take((size_t)n * 8);
    out->off = take((size_t)n);
    out->params = take(sizeof(LofParams));
    out->temp = take(temp_bytes);
    out->temp_bytes = temp_bytes;
    out->total = at;
    return cudaSuccess;
}

}  // namespace

extern "C" {

int64_t dr_lof_workspace_bytes(int64_t n) {
    if (n < 2 || n > INT32_MAX) return 0;
    LofLayout lay;
    if (lof_layout(n, &lay) != cudaSuccess) return -1;
    return (int64_t)lay.total;
}

int dr_lof_flag(dr_ctx* ctx, const double* col, int64_t n, int k, int64_t row_begin, int64_t row_count,
                uint32_t* bitmap, double* out_lof, int64_t* out_flagged, void* workspace, int64_t workspace_bytes,
                void* stream) {
    if (!ctx) return DR_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    DR_REQUIRE(ctx, n >= 0 && n <= INT32_MAX, "column length");
    DR_REQUIRE(ctx, row_begin >= 0 && row_count >= 0 && row_begin + row_count <= n, "row range");
    if (out_flagged) *out_flagged = 0;
    if (out_lof && n > 0) DR_CUDA(ctx, cudaMemsetAsync(out_lof, 0xff, (size_t)n * sizeof(double), st));  // NaN
    if (n < 2) return DR_OK;
    DR_REQUIRE(ctx, k >= 1 && k <= kLofMaxK && k <= n - 1, "1 <= k <= min(64, n - 1)");
    DR_REQUIRE(ctx, col && workspace && (bitmap || row_count == 0), "null pointer");
    LofLayout lay;
    DR_CUDA(ctx, lof_layout(n, &lay));
    DR_REQUIRE(ctx, (size_t)workspace_bytes >= lay.total, "workspace smaller than dr_lof_workspace_bytes(n)");
    char* ws = static_cast<char*>(workspace);
    auto* keys0 = reinterpret_cast<unsigned long long*>(ws + lay.keys[0]);
    auto* keys1 = reinterpret_cast<unsigned long long*>(ws + lay.keys[1]);
    auto* rows0 = reinterpret_cast<int32_t*>(ws + lay.rows[0]);
    auto* rows1 = reinterpret_cast<int32_t*>(ws + lay.rows[1]);
    auto* kdist = reinterpret_cast<double*>(ws + lay.kdist);
    auto* lrd = reinterpret_cast<double*>(ws + lay.lrd);
    auto* off = reinterpret_cast<uint8_t*>(ws + lay.off);
    auto* params = reinterpret_cast<LofParams*>(ws + lay.params);

    k_lof_keys<<<dr_grid_for(ctx, n, kLofThreads, 8), kLofThreads, 0, st>>>(col, n, keys0, rows0);
    DR_LAUNCHED(ctx);
    cub::DoubleBuffer<unsigned long long> dk(keys0, keys1);
    cub::DoubleBuffer<int32_t> dv(rows0, rows1);
    size_t temp_bytes = lay.temp_bytes;
    DR_CUDA(ctx, cub::DeviceRadixSort::SortPairs(ws + lay.temp, temp_bytes, dk, dv, (int)n, 0, 64, st));
    DR_LAUNCHED(ctx);
    const unsigned long long* keys = dk.Current();
    const int32_t* rows = dv.Current();
    double* s = reinterpret_cast<double*>(dk.Alternate());   // the sort's spare buffers hold s and perm
    int32_t* perm = dv.Alternate();
    k_lof_median<<<1, 32, 0, st>>>(keys, n, params);
    DR_LAUNCHED(ctx);
    k_lof_place<<<dr_grid_for(ctx, n, kLofThreads, 8), kLofThreads, 0, st>>>(keys, rows, n, params, s, perm);
    DR_LAUNCHED(ctx);
    const int64_t tiles = (n + kLofTile - 1) / kLofTile;
    const int grid = (int)(tiles < (int64_t)ctx->sm_count * kLofCtasPerSm ? tiles
                                                                           : (int64_t)ctx->sm_count * kLofCtasPerSm);
    k_lof_kdist<<<grid, kLofThreads, 0, st>>>(s, n, k, params, kdist, off);
    DR_LAUNCHED(ctx);
    k_lof_lrd<<<grid, kLofThreads, 0, st>>>(s, kdist, off, n, k, params, lrd);
    DR_LAUNCHED(ctx);
    k_lof_score<<<grid, kLofThreads, 0, st>>>(lrd, off, perm, n, k, row_begin, row_count, params, bitmap, out_lof);
    DR_LAUNCHED(ctx);
    if (out_flagged) {
        auto* h = reinterpret_cast<unsigned long long*>(ctx->pinned);
        DR_CUDA(ctx, cudaMemcpyAsync(h, &params->flagged, sizeof(*h), cudaMemcpyDeviceToHost, st));
        DR_CUDA(ctx, cudaStreamSynchronize(st));
        *out_flagged = (int64_t)*h;
    }
    return DR_OK;
}

}  // extern "C"
