// Shared pieces of the ADMM kernels: penalty argument pack and the elementwise proximal operators.
#pragma once
#include <math.h>

#include "common.cuh"

constexpr int kMaxPen = 4;

struct PenArgs {
    int n_pen;
    int kind[kMaxPen];
    int nn[kMaxPen];
    double p0[kMaxPen], p1[kMaxPen];
    void* aux[kMaxPen];
    void* dual[kMaxPen];
};

template <typename T>
__device__ __forceinline__ T prox_elem(T v, int kind, int nn, T p0, T p1, T rho) {
    // penalties.py:503-508 (NonNegativity), :537-542 (Box), :573-586 (L1)
    if (kind == B2_PEN_NONNEG) return v > T(0) ? v : T(0);
    if (kind == B2_PEN_BOX) return v < p0 ? p0 : (v > p1 ? p1 : v);
    // L1
    const T thr = p0 / rho;
    if (nn) {
        const T u = v - thr;
        return u > T(0) ? u : T(0);
    }
    const T a = fabs(v) - thr;
    const T m = a > T(0) ? a : T(0);
    const T sgn = v > T(0) ? T(1) : (v < T(0) ? T(-1) : T(0));
    return sgn * m;
}


// ---- row-tile helpers shared by the CTA-per-slice fused kernels (4 lanes per row, 64 rows per pass) ----
constexpr int kRowsPerPass = 64;  // 256 threads, 4 lanes per row

// Lane-owned column segment padded to a 16-byte multiple so that a row of the R x R operators can be fetched with
// 128-bit shared loads at compile-time offsets (no runtime-R address arithmetic, no bounds predicates: pad = 0).
template <typename T, int CPL>
struct RowLayout {
    static constexpr int VEC = 16 / (int)sizeof(T);
    static constexpr int CPLP = (CPL + VEC - 1) / VEC * VEC;
    static constexpr int LDM = 4 * CPLP;
    static constexpr int ROWS = 4 * CPL;
    static constexpr int ELEMS = ROWS * LDM;
};

// x[j] += sum_rr shfl(s[rr]) * M[rr][lane segment]; M in the padded RowLayout, s distributed over the 4 lanes of a row
template <typename T, int CPL>
__device__ __forceinline__ void lane_matvec(const T (&s_)[CPL], const T* __restrict__ mseg, int lane, T (&xv)[CPL]) {
    using L = RowLayout<T, CPL>;
#pragma unroll
    for (int rr = 0; rr < 4 * CPL; ++rr) {
        const T sr = __shfl_sync(0xffffffffu, s_[rr % CPL], (lane & ~3) | (rr / CPL));
        T m[L::CPLP];
#pragma unroll
        for (int v = 0; v < L::CPLP / L::VEC; ++v) *((int4*)m + v) = *((const int4*)(mseg + rr * L::LDM) + v);
#pragma unroll
        for (int j = 0; j < CPL; ++j) xv[j] = fma(sr, m[j], xv[j]);
    }
}

// Gram of a staged [64 x LDT] fp64 tile with DMMA: warp w owns the 8x8 blocks b = w, w + 8 of the NB x NB grid.
template <int NB>
__device__ __forceinline__ void tile_gram(const double* tile, int warp, int gq, int tq, double (&acc)[2][2]) {
    constexpr int LDT = 8 * NB + 2;  // 2*LDT == 4 (mod 16): conflict-free fragment reads
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int b = warp + 8 * u;
        if (b < NB * NB) {
            const int bi = b / NB, bj = b - bi * NB;
#pragma unroll
            for (int r8 = 0; r8 < kRowsPerPass / 8; ++r8) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const double* rp = tile + (r8 * 8 + h + 2 * tq) * LDT + gq;
                    dmma884(acc[u][0], acc[u][1], rp[8 * bi], rp[8 * bj]);
                }
            }
        }
    }
}

template <typename T, int NB>
__device__ __forceinline__ void store_gram(T* __restrict__ out, int R, int warp, int gq, int tq,
                                           const double (&acc)[2][2]) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int b = warp + 8 * u;
        if (b < NB * NB) {
            const int bi = b / NB, bj = b - bi * NB;
            const int i = 8 * bi + gq, j = 8 * bj + 2 * tq;
            if (i < R && j < R) out[i * R + j] = (T)acc[u][0];
            if (i < R && j + 1 < R) out[i * R + j + 1] = (T)acc[u][1];
        }
    }
}

// tensor-core row pass (pf2_mma.cu); returns -1 when it does not apply to the given shapes
int b2_pf2_rowpass_mma_try(const int64_t* row_off, int n_groups, int R, const void* Y, const void* A, const void* rho,
                           const void* Minv, const PenArgs& pa, int deferred, const void* Wmat, const void* Delta,
                           void* x, void* w_out, int ldw, void* S_out, void* BtB_out, int dtype, cudaStream_t st);

// second-generation tensor-core row pass (pf2_rowpass_v2.cu: fp64, R % 4 == 0, deferred prox, at most one
// non-negativity companion); returns -1 when it does not apply
int b2_pf2_rowpass_v2_try(const int64_t* row_off, int n_groups, int R, const void* Y, const void* A, const void* rho,
                          const void* Minv, const PenArgs& pa, int deferred, const void* Wmat, const void* Delta,
                          void* x, void* w_out, int ldw, void* S_out, void* BtB_out, double* stats_part, int dtype,
                          cudaStream_t st);
int b2_pf2_rowpass_v2_applies(int R, int dtype, int n_pen, int companion_kind, int deferred);

// tensor-core PARAFAC2 gap reduction (pf2_gap_mma.cu); returns -1 when it does not apply
int b2_pf2_gap_mma_try(const void* V, const void* x, const int64_t* row_off, int n_groups, int R, const void* Wmat,
                       const void* Delta, double* part, int dtype, cudaStream_t st);

// tensor-core fused row-local ADMM loop (admm_mma.cu); returns -1 when it does not apply
int b2_admm_local_mma_try(const int64_t* row_off, int n_groups, int R, const void* rhs, const void* rhs_scale,
                          const void* rho, const void* Minv, const PenArgs& pa, int n_inner, void* x, void* w_out,
                          int ldw, void* BtB_out, int dtype, cudaStream_t st);

// host: validate and pack the caller's descriptors
inline int b2_pack_penalties(const b2_penalty_desc* pens, int n_pen, PenArgs* pa) {
    B2_REQUIRE(n_pen >= 0 && n_pen <= kMaxPen, "at most %d penalties per mode are supported (got %d)", kMaxPen, n_pen);
    pa->n_pen = n_pen;
    for (int p = 0; p < n_pen; ++p) {
        B2_REQUIRE(pens[p].kind >= B2_PEN_NONNEG && pens[p].kind <= B2_PEN_TEMPORAL, "unknown penalty kind %d",
                   pens[p].kind);
        B2_REQUIRE(pens[p].aux && pens[p].dual, "penalty %d: aux/dual pointers must be set", p);
        pa->kind[p] = pens[p].kind;
        pa->nn[p] = pens[p].non_negativity;
        pa->p0[p] = pens[p].p0;
        pa->p1[p] = pens[p].p1;
        pa->aux[p] = pens[p].aux;
        pa->dual[p] = pens[p].dual;
    }
    return B2_OK;
}
