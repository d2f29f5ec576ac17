// TemporalSmoothnessPenalty: g(B_0..B_{I-1}) = lam * sum_{i>=1} ||B_i - B_{i-1}||_F^2 over the slice order.
//   b2_prox_temporal          : (diag(rho) + 2 lam L) z = rho o v for every position (j, r) of the slices, L the
//                               path-graph Laplacian; aux = z, dual = V - z (V arrives in `dual`)
//   b2_prox_temporal_serial   : the same solve, one thread per position running Thomas over all I slices (baseline)
//   b2_temporal_norm          : lam * sum_i ||B_i - B_{i-1}||^2, per-pair partials summed in a fixed order
//
// The tridiagonal matrix T = diag(rho) + 2 lam L is the same for all J*R positions, so everything that depends only on
// T is computed once per call (O(I) scalars) and the per-position work is streaming FMAs.  Partition (spike) solve:
//   setup    : per chunk q of kChunk slices the Thomas factors of the chunk block T_q (r_k = rho_k / den_k and
//              w_k = 2 lam / den_k) and the spike vectors alpha_q = T_q^-1 (2 lam e_first), beta_q = T_q^-1 (2 lam
//              e_last); then the multipliers of the reduced 2 x 2 block-tridiagonal system in the chunk ends
//   phase 1  : per (chunk, position) the chunk-local solve with zero outer boundaries in registers; only its two end
//              values are written (fp64, L2-resident)
//   phase 2  : per position two FMA sweeps over the chunk ends solve the reduced system
//   phase 3  : per (chunk, position) the chunk-local solve again, plus alpha_q z_left + beta_q z_right; aux and dual
//              are written in the same pass
// Traffic: V read twice, aux and dual written once: 4 N R sizeof(T) (the reduced system's 2 N R / kChunk doubles stay
// in L2).  Sharded runs (stage 1 / 2): every rank is one top-level block, solved with the same machinery; its ends and
// spike ends go through one all-reduce, and every rank solves the small 2 * world system identically.
// All sums run in fp64 (fp32 data too), in a fixed order, without atomics: two launches give the same bits.
#include "common.cuh"

namespace {

constexpr int kChunk = 32;     // slices per chunk: the chunk solve keeps kChunk doubles per thread in registers
constexpr int kThreads = 128;  // positions per block of the chunk passes
constexpr int kRankCoef = 7;   // per rank of a sharded solve: a0, a1, s00, s10, sb0, sb1, holds-slices flag

// workspace layout (doubles)
struct TemporalWs {
    double *r, *w, *alpha, *beta;  // I each
    double *a, *b, *s, *sb;        // 2Q each: chunk-end spike values, S_q^-1 = [[s0, 0], [s1, 1]], S_q^-1 b_q
    double *aR, *bR;               // 2Q each: ends of the rank-level spike vectors at every chunk end (sharded)
    double *bnd;                   // 2 Q P: chunk-end values, row 2q = first slice of chunk q, row 2q+1 = last
    double *zl, *zr;               // P each: the neighbours' boundary values of this rank (sharded)
    double *rank_coef;             // kRankCoef * world
};

long long n_chunks(long long I) { return (I + kChunk - 1) / kChunk; }

size_t ws_doubles(long long I, long long P, int world) {
    const long long Q = n_chunks(I);
    return (size_t)(4 * I + 12 * Q + 2 * Q * P + 2 * P + (long long)kRankCoef * world);
}

TemporalWs carve(void* ws, long long I, long long P) {
    const long long Q = n_chunks(I);
    double* p = (double*)ws;
    TemporalWs t;
    t.r = p; p += I;
    t.w = p; p += I;
    t.alpha = p; p += I;
    t.beta = p; p += I;
    t.a = p; p += 2 * Q;
    t.b = p; p += 2 * Q;
    t.s = p; p += 2 * Q;
    t.sb = p; p += 2 * Q;
    t.aR = p; p += 2 * Q;
    t.bR = p; p += 2 * Q;
    t.bnd = p; p += 2 * Q * P;
    t.zl = p; p += P;
    t.zr = p; p += P;
    t.rank_coef = p;
    return t;
}

// ---------------------------------------------------------------------------------------------------------------
// setup (position-independent, O(I))
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void temporal_setup_chunks_kernel(const T* __restrict__ rho, int rho_stride, double lam, long long I,
                                             long long chunk, long long Q, int has_left, int has_right, TemporalWs t) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    const long long s = q * chunk, n = (I - s < chunk ? I - s : chunk), e = s + n;
    const double tl = 2.0 * lam;
    // Thomas factors of the chunk block: den_s = D_s, den_k = D_k - 2 lam w_{k-1}; the diagonal D_k = rho_k + 2 lam
    // deg_k uses the degree in the WHOLE slice graph (a rank's outer neighbours included)
    double w_prev = 0.0;
    for (long long k = s; k < e; ++k) {
        const double rk = (double)rho[k * rho_stride];
        const int deg = ((k > 0 || has_left) ? 1 : 0) + ((k < I - 1 || has_right) ? 1 : 0);
        const double den = rk + tl * deg - (k > s ? tl * w_prev : 0.0);
        t.r[k] = rk / den;  // I = 1 without neighbours: rho / rho = 1 exactly, the identity prox
        t.w[k] = tl / den;
        w_prev = t.w[k];
    }
    // alpha = T_q^-1 (2 lam e_first): forward d_s = w_s, d_k = w_k d_{k-1}; backward z_k = d_k + w_k z_{k+1}
    double d = 0.0;
    for (long long k = s; k < e; ++k) {
        d = (k == s) ? t.w[k] : t.w[k] * d;
        t.alpha[k] = d;
    }
    for (long long k = e - 2; k >= s; --k) t.alpha[k] += t.w[k] * t.alpha[k + 1];
    // beta = T_q^-1 (2 lam e_last): forward leaves d_{e-1} = w_{e-1}; backward z_k = w_k z_{k+1}
    t.beta[e - 1] = t.w[e - 1];
    for (long long k = e - 2; k >= s; --k) t.beta[k] = t.w[k] * t.beta[k + 1];
    // coupling of the reduced system: no left neighbour for chunk 0, no right neighbour for the last chunk
    t.a[2 * q] = q > 0 ? t.alpha[s] : 0.0;
    t.a[2 * q + 1] = q > 0 ? t.alpha[e - 1] : 0.0;
    t.b[2 * q] = q < Q - 1 ? t.beta[s] : 0.0;
    t.b[2 * q + 1] = q < Q - 1 ? t.beta[e - 1] : 0.0;
}

// Reduced system in the chunk ends w_q = (first_q, last_q):  w_q - a_q last_{q-1} - b_q first_{q+1} = y_q.
// Block Thomas with identity diagonal blocks: S_q = I - c_q a_q e1^T (c_q = (S_{q-1}^-1 b_{q-1})[1]) is lower
// triangular, S_q^-1 = [[s0, 0], [s1, 1]]; per position then  h_q = S_q^-1 (y_q + a_q h_{q-1}[1]),
// w_q = h_q + (S_q^-1 b_q) first_{q+1}.
__device__ void reduced_factor(const double* a, const double* b, long long Q, double* s, double* sb) {
    double c = 0.0;
    for (long long q = 0; q < Q; ++q) {
        const double s0 = 1.0 / (1.0 - c * a[2 * q]);
        const double s1 = c * a[2 * q + 1] * s0;
        s[2 * q] = s0;
        s[2 * q + 1] = s1;
        sb[2 * q] = s0 * b[2 * q];
        sb[2 * q + 1] = s1 * b[2 * q] + b[2 * q + 1];
        c = sb[2 * q + 1];
    }
}

// one right-hand side of the reduced system (y given at chunk q_rhs only), solved serially: the chunk ends of the
// rank-level spike vectors
__device__ void reduced_solve_one(const double* a, const double* s, const double* sb, long long Q, long long q_rhs,
                                  double y0, double y1, double* out) {
    double h1 = 0.0;
    for (long long q = 0; q < Q; ++q) {
        const double g0 = (q == q_rhs ? y0 : 0.0) + a[2 * q] * h1;
        const double g1 = (q == q_rhs ? y1 : 0.0) + a[2 * q + 1] * h1;
        out[2 * q] = s[2 * q] * g0;
        out[2 * q + 1] = s[2 * q + 1] * g0 + g1;
        h1 = out[2 * q + 1];
    }
    double f_next = 0.0;
    for (long long q = Q - 1; q >= 0; --q) {
        out[2 * q] += sb[2 * q] * f_next;
        out[2 * q + 1] += sb[2 * q + 1] * f_next;
        f_next = out[2 * q];
    }
}

__global__ void temporal_setup_reduced_kernel(long long I, long long Q, TemporalWs t, double* xrow, long long P) {
    reduced_factor(t.a, t.b, Q, t.s, t.sb);
    if (xrow != nullptr) {
        // spike vectors of the whole local block: T_loc^-1 (2 lam e_first) has the local solution alpha_0 in chunk 0
        // and zero elsewhere, T_loc^-1 (2 lam e_last) has beta_{Q-1} in the last chunk
        const long long sl = (Q - 1) * kChunk;
        reduced_solve_one(t.a, t.s, t.sb, Q, 0, t.alpha[0], t.alpha[(I < kChunk ? I : kChunk) - 1], t.aR);
        reduced_solve_one(t.a, t.s, t.sb, Q, Q - 1, t.beta[sl], t.beta[I - 1], t.bR);
        xrow[2 * P + 0] = t.aR[0];
        xrow[2 * P + 1] = t.aR[2 * Q - 1];
        xrow[2 * P + 2] = t.bR[0];
        xrow[2 * P + 3] = t.bR[2 * Q - 1];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// phases 1 and 3: one thread per (chunk, position); the kChunk values of a chunk stay in registers
// ---------------------------------------------------------------------------------------------------------------
template <typename T, bool FINISH>
__global__ void __launch_bounds__(kThreads)
temporal_chunk_kernel(T* __restrict__ aux, T* __restrict__ dual, long long I, long long P, long long Q, TemporalWs t,
                      int sharded) {
    const long long p = (long long)blockIdx.x * kThreads + threadIdx.x;
    if (p >= P) return;
    for (long long q = blockIdx.y; q < Q; q += gridDim.y) {
        const long long s = q * kChunk;
        const int n = (int)(I - s < kChunk ? I - s : kChunk);
        const T* V = dual + s * P + p;
        double y[kChunk];
        double d = 0.0;
#pragma unroll
        for (int k = 0; k < kChunk; ++k) {
            y[k] = 0.0;
            if (k < n) {
                d = __ldg(t.r + s + k) * (double)V[k * P] + __ldg(t.w + s + k) * d;
                y[k] = d;
            }
        }
        if constexpr (!FINISH) {  // only the two end values: d is the last one, the backward sweep ends at the first
            double z = d;
#pragma unroll
            for (int k = kChunk - 2; k >= 0; --k) {
                if (k < n - 1) z = y[k] + __ldg(t.w + s + k) * z;
            }
            t.bnd[(2 * q) * P + p] = z;
            t.bnd[(2 * q + 1) * P + p] = d;
        } else {
#pragma unroll
            for (int k = kChunk - 2; k >= 0; --k) {
                if (k < n - 1) y[k] += __ldg(t.w + s + k) * y[k + 1];
            }
            // true values of the neighbouring slices: chunk ends of the reduced solution (with the rank's outer
            // boundary values added through the rank-level spike vectors when sharded)
            const double zl = sharded ? t.zl[p] : 0.0, zr = sharded ? t.zr[p] : 0.0;
            double left = zl, right = zr;
            if (q > 0) {
                const long long i = 2 * (q - 1) + 1;
                left = t.bnd[i * P + p];
                if (sharded) left += t.aR[i] * zl + t.bR[i] * zr;
            }
            if (q < Q - 1) {
                const long long i = 2 * (q + 1);
                right = t.bnd[i * P + p];
                if (sharded) right += t.aR[i] * zl + t.bR[i] * zr;
            }
            T* Au = aux + s * P + p;
            T* Du = dual + s * P + p;
#pragma unroll
            for (int k = 0; k < kChunk; ++k) {
                if (k < n) {
                    const double z = y[k] + __ldg(t.alpha + s + k) * left + __ldg(t.beta + s + k) * right;
                    const T zt = (T)z;
                    const T v = Du[k * P];
                    Au[k * P] = zt;
                    Du[k * P] = v - zt;
                }
            }
        }
    }
}

// phase 2: per position, the two sweeps of the reduced system (in place in bnd); stage 1 also writes the local
// solution's end values into this rank's exchange row
__global__ void __launch_bounds__(256)
temporal_reduced_kernel(long long P, long long Q, TemporalWs t, double* __restrict__ xrow) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    double* B = t.bnd + p;
    double h1 = 0.0;
#pragma unroll 4
    for (long long q = 0; q < Q; ++q) {
        const double g0 = B[(2 * q) * P] + __ldg(t.a + 2 * q) * h1;
        const double g1 = B[(2 * q + 1) * P] + __ldg(t.a + 2 * q + 1) * h1;
        const double h0 = __ldg(t.s + 2 * q) * g0;
        h1 = __ldg(t.s + 2 * q + 1) * g0 + g1;
        B[(2 * q) * P] = h0;
        B[(2 * q + 1) * P] = h1;
    }
    double f_next = 0.0;
#pragma unroll 4
    for (long long q = Q - 1; q >= 0; --q) {
        const double w0 = B[(2 * q) * P] + __ldg(t.sb + 2 * q) * f_next;
        const double w1 = B[(2 * q + 1) * P] + __ldg(t.sb + 2 * q + 1) * f_next;
        B[(2 * q) * P] = w0;
        B[(2 * q + 1) * P] = w1;
        f_next = w0;
    }
    if (xrow != nullptr) {
        xrow[p] = B[0];
        xrow[P + p] = B[(2 * Q - 1) * P];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// sharded runs: the reduced system over the ranks.  Exchange row r (width 2P + 4, all-reduced, zero for a rank
// without slices): [first-slice values of the rank's local solution (P), last-slice values (P), alpha_first,
// alpha_last, beta_first, beta_last].  A rank holds slices iff alpha_first > 0 (T^-1 of an M-matrix is positive).
// ---------------------------------------------------------------------------------------------------------------
__global__ void temporal_rank_factor_kernel(const double* __restrict__ xch, int world, long long P,
                                            double* __restrict__ coef) {
    const long long W = 2 * P + 4;
    int first = -1, last = -1;
    for (int r = 0; r < world; ++r)
        if (xch[r * W + 2 * P] > 0.0) {
            if (first < 0) first = r;
            last = r;
        }
    double c = 0.0;
    for (int r = 0; r < world; ++r) {
        double* cf = coef + kRankCoef * r;
        const double* x = xch + r * W + 2 * P;
        const bool on = first >= 0 && x[0] > 0.0;
        const double a0 = on && r != first ? x[0] : 0.0, a1 = on && r != first ? x[1] : 0.0;
        const double b0 = on && r != last ? x[2] : 0.0, b1 = on && r != last ? x[3] : 0.0;
        cf[0] = a0;
        cf[1] = a1;
        cf[6] = on ? 1.0 : 0.0;
        if (!on) continue;
        const double s0 = 1.0 / (1.0 - c * a0), s1 = c * a1 * s0;
        cf[2] = s0;
        cf[3] = s1;
        cf[4] = s0 * b0;
        cf[5] = s1 * b0 + b1;
        c = cf[5];
    }
}

__global__ void __launch_bounds__(256)
temporal_rank_solve_kernel(double* __restrict__ xch, int world, int rank, long long P,
                           const double* __restrict__ coef, double* __restrict__ zl, double* __restrict__ zr) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const long long W = 2 * P + 4;
    double h1 = 0.0;
    for (int r = 0; r < world; ++r) {  // in place in this position's entries of the (rank-local copy of the) rows
        const double* cf = coef + kRankCoef * r;
        if (cf[6] == 0.0) continue;
        double* x = xch + r * W + p;
        const double g0 = x[0] + cf[0] * h1, g1 = x[P] + cf[1] * h1;
        x[0] = cf[2] * g0;
        h1 = cf[3] * g0 + g1;
        x[P] = h1;
    }
    double f_next = 0.0, left = 0.0, right = 0.0;
    for (int r = world - 1; r >= 0; --r) {
        const double* cf = coef + kRankCoef * r;
        if (cf[6] == 0.0) continue;
        double* x = xch + r * W + p;
        const double w0 = x[0] + cf[4] * f_next, w1 = x[P] + cf[5] * f_next;
        if (r < rank) {
            left = w1;  // last slice of the nearest rank with slices before this one
            break;
        }
        if (r > rank) right = w0;  // descending: ends as the first slice of the nearest rank after this one
        f_next = w0;
    }
    zl[p] = left;
    zr[p] = right;
}

// ---------------------------------------------------------------------------------------------------------------
// baseline: one thread per position, Thomas over all I slices (forward values parked in aux)
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
temporal_serial_kernel(T* __restrict__ aux, T* __restrict__ dual, long long I, long long P, const double* __restrict__ r,
                       const double* __restrict__ w) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    double d = 0.0;
    for (long long k = 0; k < I; ++k) {
        d = __ldg(r + k) * (double)dual[k * P + p] + __ldg(w + k) * d;
        aux[k * P + p] = (T)d;
    }
    double z = d;
    for (long long k = I - 1; k >= 0; --k) {
        if (k < I - 1) z = (double)aux[k * P + p] + __ldg(w + k) * z;
        const T zt = (T)z;
        aux[k * P + p] = zt;
        dual[k * P + p] = dual[k * P + p] - zt;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// penalty value
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
temporal_norm_kernel(const T* __restrict__ x, long long P, const double* __restrict__ xch, int rank,
                     double* __restrict__ part) {
    __shared__ double scratch[32];
    const long long i = blockIdx.x;  // pair (i - 1, i); pair 0 = (last slice of the previous rank, slice 0)
    const T* cur = x + i * P;
    double acc = 0.0;
    if (i > 0) {
        const T* prev = cur - P;
        for (long long e = threadIdx.x; e < P; e += blockDim.x) {
            const double dlt = (double)cur[e] - (double)prev[e];
            acc += dlt * dlt;
        }
    } else if (xch != nullptr) {
        // exchange rows of width P + 1: [last slice of rank r, 1 if rank r holds slices]
        const double* prev = nullptr;
        for (int r = rank - 1; r >= 0 && prev == nullptr; --r)
            if (xch[(long long)r * (P + 1) + P] != 0.0) prev = xch + (long long)r * (P + 1);
        if (prev != nullptr)
            for (long long e = threadIdx.x; e < P; e += blockDim.x) {
                const double dlt = (double)cur[e] - prev[e];
                acc += dlt * dlt;
            }
    }
    acc = block_sum(acc, scratch);
    if (threadIdx.x == 0) part[i] = acc;
}

__global__ void __launch_bounds__(256)
temporal_norm_finish_kernel(const double* __restrict__ part, long long n, double lam, double* __restrict__ out) {
    __shared__ double scratch[32];
    double acc = 0.0;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) acc += part[i];
    acc = block_sum(acc, scratch);
    if (threadIdx.x == 0) out[0] = lam * acc;
}

int check_common(const char* fn, long long I, long long P, double lam) {
    B2_REQUIRE(I >= 0 && P >= 0, "%s: bad shape (n_slices %lld, n_pos %lld)", fn, I, P);
    B2_REQUIRE(lam > 0.0, "%s: smoothness_reg must be positive (got %g)", fn, lam);
    return B2_OK;
}

// after the empty-shape return: a rank without slices may pass a NULL (zero-size) rho
int check_operands(const char* fn, const void* aux, const void* dual, const void* rho, int rho_stride, const void* ws) {
    B2_REQUIRE(rho != nullptr && (rho_stride == 0 || rho_stride == 1), "%s: rho (device) with stride 0 or 1", fn);
    B2_REQUIRE(aux != nullptr && dual != nullptr && ws != nullptr, "%s: null aux/dual/workspace", fn);
    return B2_OK;
}

}  // namespace

extern "C" {

size_t b2_prox_temporal_workspace_bytes(long long n_slices, long long n_pos, int world) {
    if (n_slices < 0 || n_pos < 0 || world < 1) return 0;
    return sizeof(double) * ws_doubles(n_slices, n_pos, world);
}

int b2_prox_temporal(void* aux, void* dual, long long n_slices, long long n_pos, const void* rho, int rho_stride,
                     double lam, int stage, int has_left, int has_right, double* xch, int world, int rank, int dtype,
                     void* ws, size_t ws_bytes, void* stream) {
    const long long I = n_slices, P = n_pos;
    if (int rc = check_common("b2_prox_temporal", I, P, lam)) return rc;
    B2_REQUIRE(stage >= 0 && stage <= 2, "b2_prox_temporal: stage %d outside 0..2", stage);
    B2_REQUIRE(stage == 0 ? (world == 1 && !has_left && !has_right)
                          : (xch != nullptr && world >= 1 && rank >= 0 && rank < world),
               "b2_prox_temporal: stage %d with world %d, rank %d, neighbours %d/%d and exchange buffer %p", stage,
               world, rank, has_left, has_right, (void*)xch);
    if (I == 0 || P == 0) return B2_OK;  // a rank without slices still takes part in the caller's all-reduce
    if (int rc = check_operands("b2_prox_temporal", aux, dual, rho, rho_stride, ws)) return rc;
    B2_REQUIRE(ws_bytes >= b2_prox_temporal_workspace_bytes(I, P, world),
               "b2_prox_temporal workspace too small (%zu < %zu bytes)", ws_bytes,
               b2_prox_temporal_workspace_bytes(I, P, world));
    cudaStream_t st = (cudaStream_t)stream;
    const long long Q = n_chunks(I);
    TemporalWs t = carve(ws, I, P);
    const long long W = 2 * P + 4;
    const dim3 grid((unsigned)((P + kThreads - 1) / kThreads), (unsigned)(Q < 65535 ? Q : 65535));
    const unsigned pblocks = (unsigned)((P + 255) / 256);
    if (stage <= 1) {
        double* xrow = stage == 1 ? xch + (long long)rank * W : nullptr;
        B2_DISPATCH_DTYPE(dtype, {
            temporal_setup_chunks_kernel<T><<<(unsigned)((Q + 127) / 128), 128, 0, st>>>(
                (const T*)rho, rho_stride, lam, I, kChunk, Q, has_left, has_right, t);
            B2_LAUNCH_CHECK();
            temporal_setup_reduced_kernel<<<1, 1, 0, st>>>(I, Q, t, xrow, P);
            B2_LAUNCH_CHECK();
            temporal_chunk_kernel<T, false><<<grid, kThreads, 0, st>>>((T*)aux, (T*)dual, I, P, Q, t, 0);
            B2_LAUNCH_CHECK();
            temporal_reduced_kernel<<<pblocks, 256, 0, st>>>(P, Q, t, xrow);
            B2_LAUNCH_CHECK();
        });
        if (stage == 1) return B2_OK;
    } else {
        temporal_rank_factor_kernel<<<1, 1, 0, st>>>(xch, world, P, t.rank_coef);
        B2_LAUNCH_CHECK();
        temporal_rank_solve_kernel<<<pblocks, 256, 0, st>>>(xch, world, rank, P, t.rank_coef, t.zl, t.zr);
        B2_LAUNCH_CHECK();
    }
    B2_DISPATCH_DTYPE(dtype, {
        temporal_chunk_kernel<T, true><<<grid, kThreads, 0, st>>>((T*)aux, (T*)dual, I, P, Q, t, stage == 2);
        B2_LAUNCH_CHECK();
    });
    return B2_OK;
}

int b2_prox_temporal_serial(void* aux, void* dual, long long n_slices, long long n_pos, const void* rho,
                            int rho_stride, double lam, int dtype, void* ws, size_t ws_bytes, void* stream) {
    const long long I = n_slices, P = n_pos;
    if (int rc = check_common("b2_prox_temporal_serial", I, P, lam)) return rc;
    if (I == 0 || P == 0) return B2_OK;
    if (int rc = check_operands("b2_prox_temporal_serial", aux, dual, rho, rho_stride, ws)) return rc;
    B2_REQUIRE(ws_bytes >= b2_prox_temporal_workspace_bytes(I, P, 1),
               "b2_prox_temporal_serial workspace too small (%zu < %zu bytes)", ws_bytes,
               b2_prox_temporal_workspace_bytes(I, P, 1));
    cudaStream_t st = (cudaStream_t)stream;
    TemporalWs t = carve(ws, I, P);
    B2_DISPATCH_DTYPE(dtype, {
        // the Thomas factors of the whole system: one "chunk" of I slices
        temporal_setup_chunks_kernel<T><<<1, 1, 0, st>>>((const T*)rho, rho_stride, lam, I, I, 1, 0, 0, t);
        B2_LAUNCH_CHECK();
        temporal_serial_kernel<T><<<(unsigned)((P + 255) / 256), 256, 0, st>>>((T*)aux, (T*)dual, I, P, t.r, t.w);
        B2_LAUNCH_CHECK();
    });
    return B2_OK;
}

int b2_temporal_norm(const void* x, long long n_slices, long long n_pos, double lam, const double* xch, int rank,
                     double* out, double* part, int dtype, void* stream) {
    const long long I = n_slices, P = n_pos;
    B2_REQUIRE(I >= 0 && P >= 0, "b2_temporal_norm: bad shape (n_slices %lld, n_pos %lld)", I, P);
    B2_REQUIRE(lam > 0.0, "b2_temporal_norm: smoothness_reg must be positive (got %g)", lam);
    B2_REQUIRE(out != nullptr, "b2_temporal_norm: null out");
    B2_REQUIRE(xch == nullptr || rank >= 0, "b2_temporal_norm: rank %d", rank);
    cudaStream_t st = (cudaStream_t)stream;
    if (I == 0 || P == 0) {
        B2_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(double), st));
        return B2_OK;
    }
    B2_REQUIRE(x != nullptr && part != nullptr, "b2_temporal_norm needs x and n_slices doubles of scratch");
    B2_REQUIRE(I < 2147483647LL, "b2_temporal_norm: %lld slices", I);
    B2_DISPATCH_DTYPE(dtype, {
        temporal_norm_kernel<T><<<(unsigned)I, 256, 0, st>>>((const T*)x, P, xch, rank, part);
        B2_LAUNCH_CHECK();
    });
    temporal_norm_finish_kernel<<<1, 256, 0, st>>>(part, I, lam, out);
    B2_LAUNCH_CHECK();
    return B2_OK;
}

}  // extern "C"
