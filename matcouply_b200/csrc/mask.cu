// Missing-entry refill for masked fitting (EM with one refill per outer iteration, DESIGN.md §10):
//   b2_mask_refill : X[n][k] <- (B[n] o A[g]) . C[k] for every missing (n, k); Y[n] += sum_k d_k C[k]; sums for the loss
//
// Bandwidth kernel over a CSR list of missing entries.  One warp owns a row (lane r holds column r of the rank, R <= 32):
// w_r = B[n][r] A[g][r] is read once, the row's missing columns are walked in chunks of 32 (lane j gathers column j of
// the chunk and its current fill), and for every entry the warp reads the row C[k] (L2-resident, K x R <= 2 MB at
// R = 32), forms xhat with a butterfly sum and adds d C[k] to the Y-row correction held in registers.  No atomics:
// every lane sums its entries in row order, warps and blocks reduce in a fixed order, a one-block kernel adds the block
// partials into out[0:2] — bit-reproducible runs.
#include "common.cuh"

namespace {

constexpr int kThreads = 256;  // 8 rows in flight per block
constexpr int kWarps = kThreads / 32;

int refill_blocks(long long n_rows) {
    const long long want = (n_rows + kWarps - 1) / kWarps;
    const long long cap = 4LL * b2_num_sms();  // 4 resident blocks per SM at <= 64 registers: 32 rows in flight
    return (int)(want < 1 ? 1 : (want < cap ? want : cap));
}

template <typename T>
__global__ void __launch_bounds__(kThreads) mask_refill_kernel(T* __restrict__ X, long long n_rows, int ldx,
                                                               const int64_t* __restrict__ row_ptr,
                                                               const int32_t* __restrict__ miss_col,
                                                               const int32_t* __restrict__ gor, const T* __restrict__ A,
                                                               const T* __restrict__ B, const T* __restrict__ C, int R,
                                                               T* __restrict__ Y, double* __restrict__ part) {
    __shared__ double scratch[32];
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * kWarps + (threadIdx.x >> 5);
    const long long n_warps = (long long)gridDim.x * kWarps;
    const bool col = lane < R;
    double sq_miss = 0.0, d_norm = 0.0;  // this lane's share of out[0], out[1]
    for (long long n = warp0; n < n_rows; n += n_warps) {
        const long long p0 = __ldg(row_ptr + n), p1 = __ldg(row_ptr + n + 1);
        if (p0 == p1) continue;  // no missing entry: one row_ptr read
        const int g = __ldg(gor + n);
        const double w = col ? (double)__ldg(B + n * R + lane) * (double)__ldg(A + (long long)g * R + lane) : 0.0;
        double ycorr = 0.0;
        T* xrow = X + n * (long long)ldx;
        for (long long p = p0; p < p1; p += 32) {
            const int cnt = (int)(p1 - p < 32 ? p1 - p : 32);
            int kj = 0;
            double xj = 0.0;
            if (lane < cnt) {
                kj = __ldg(miss_col + p + lane);
                xj = (double)xrow[kj];
            }
            double mine = 0.0;
#pragma unroll 4
            for (int j = 0; j < cnt; ++j) {
                const int k = __shfl_sync(0xffffffffu, kj, j);
                const double x = __shfl_sync(0xffffffffu, xj, j);
                const double c = col ? (double)__ldg(C + (long long)k * R + lane) : 0.0;
                const double xhat = (double)(T)warp_sum(w * c);  // every lane holds the same sum (butterfly)
                ycorr += (xhat - x) * c;
                if (lane == j) mine = xhat;
            }
            if (lane < cnt) {
                const double d = mine - xj;
                sq_miss += d * d;
                d_norm += mine * mine - xj * xj;
                xrow[kj] = (T)mine;
            }
        }
        if (Y != nullptr && col) Y[n * R + lane] = (T)((double)Y[n * R + lane] + ycorr);
    }
    sq_miss = block_sum(sq_miss, scratch);
    d_norm = block_sum(d_norm, scratch);
    if (threadIdx.x == 0) {
        part[blockIdx.x] = sq_miss;
        part[gridDim.x + blockIdx.x] = d_norm;
    }
}

__global__ void mask_refill_finish_kernel(const double* __restrict__ part, int n, double* __restrict__ out) {
    __shared__ double scratch[32];
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        a += part[i];
        b += part[n + i];
    }
    a = block_sum(a, scratch);
    b = block_sum(b, scratch);
    if (threadIdx.x == 0) {
        out[0] += a;
        out[1] += b;
    }
}

}  // namespace

extern "C" {

size_t b2_mask_refill_workspace_bytes(long long n_rows) { return 2 * sizeof(double) * (size_t)refill_blocks(n_rows); }

int b2_mask_refill(void* X, long long n_rows, int K, int ldx, const int64_t* miss_row_ptr, const int32_t* miss_col,
                   const int32_t* group_of_row, const void* A, const void* B, const void* C, int R, void* Y,
                   double* out, int dtype, void* ws, size_t ws_bytes, void* stream) {
    B2_REQUIRE(R >= 1 && R <= B2_MAX_RANK, "b2_mask_refill: rank %d outside 1..%d", R, B2_MAX_RANK);
    B2_REQUIRE(n_rows >= 0 && K >= 0 && ldx >= K, "b2_mask_refill: bad shape (n_rows %lld, K %d, ldx %d)", n_rows, K,
               ldx);
    if (n_rows == 0) return B2_OK;
    const int blocks = refill_blocks(n_rows);
    B2_REQUIRE(ws_bytes >= 2 * sizeof(double) * (size_t)blocks, "b2_mask_refill workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    B2_DISPATCH_DTYPE(dtype, mask_refill_kernel<T><<<blocks, kThreads, 0, st>>>(
                                 (T*)X, n_rows, ldx, miss_row_ptr, miss_col, group_of_row, (const T*)A, (const T*)B,
                                 (const T*)C, R, (T*)Y, (double*)ws));
    B2_LAUNCH_CHECK();
    mask_refill_finish_kernel<<<1, 256, 0, st>>>((const double*)ws, blocks, out);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

}  // extern "C"
