// dcr_common.cuh — shared device/host helpers of libdcr (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/dcr.h"

namespace dcr {

// ------------------------------------------------------------------------------------------------------------
// error reporting (thread-local message behind dcr_last_error())
// ------------------------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define DCR_CUDA(call)                                                        \
    do {                                                                      \
        cudaError_t e__ = (call);                                             \
        if (e__ != cudaSuccess) return dcr::cuda_fail(e__, #call, __FILE__, __LINE__); \
    } while (0)

#define DCR_LAUNCH_CHECK() DCR_CUDA(cudaGetLastError())

constexpr int MAX_DEVICES = 64;   // per-device host-side state (streams, function attributes) is indexed by ordinal
int current_device();
int sm_count();

constexpr unsigned FULL = 0xffffffffu;

// ------------------------------------------------------------------------------------------------------------
// A read-only view of an adjacency structure with sorted rows.  The static CSR (rowptr) and the SDRF arena
// (row start / length arrays) are both expressed this way: row v occupies col[start[v] .. start[v]+len(v)).
// ------------------------------------------------------------------------------------------------------------
struct GraphView {
    const int32_t* start;  // row offsets
    const int32_t* len;    // row lengths, or nullptr for a packed CSR (len = start[v+1]-start[v])
    const int32_t* col;    // sorted neighbour ids
    __device__ __forceinline__ int begin(int v) const { return start[v]; }
    __device__ __forceinline__ int degree(int v) const { return len ? len[v] : start[v + 1] - start[v]; }
};

// position of `key` in the sorted range col[lo, lo+n), or -1
__device__ __forceinline__ int find_sorted(const int32_t* __restrict__ col, int lo, int n, int key) {
    int a = 0, b = n;
    while (a < b) {
        int m = (a + b) >> 1;
        int v = col[lo + m];
        if (v < key) a = m + 1; else b = m;
    }
    return (a < n && col[lo + a] == key) ? lo + a : -1;
}

// lower bound: first index t in [0,n) with col[lo+t] >= key
__device__ __forceinline__ int lower_bound(const int32_t* __restrict__ col, int lo, int n, int key) {
    int a = 0, b = n;
    while (a < b) {
        int m = (a + b) >> 1;
        if (col[lo + m] < key) a = m + 1; else b = m;
    }
    return a;
}

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = max(v, __shfl_xor_sync(FULL, v, o));
    return v;
}

// Warp-cooperative |N(a) ∩ N(b)|: lanes take elements of the shorter row and binary-search the longer one.
__device__ __forceinline__ int warp_intersect_count(const GraphView& g, int a, int b, int lane) {
    int da = g.degree(a), db = g.degree(b);
    int sa = g.begin(a), sb = g.begin(b);
    if (da > db) { int t = da; da = db; db = t; t = sa; sa = sb; sb = t; }
    int c = 0;
    for (int t = lane; t < da; t += 32) c += find_sorted(g.col, sb, db, g.col[sa + t]) >= 0;
    return warp_sum(c);
}

// ------------------------------------------------------------------------------------------------------------
// The closing formula of the reference's numba kernels exactly as the compiled PTX evaluates it
// (curvature/bfc_cuda.py:46-48 and :139-141; dataflow in SURVEY.md App. A.3): fp64 round-to-nearest operations,
// one fp32 store, then — when lambda > 0 — a second fp64 add onto the widened fp32 value and a second store.
// Intrinsics with explicit rounding stop nvcc from contracting or re-associating anything.
//   d_max, d_min : the fp32 degrees (exact small integers)       a2 : A2[i,j] (fp32-exact integer)
//   a_xy         : A[i,j] in {0,1}                               sharp, lam : integer counts
// ------------------------------------------------------------------------------------------------------------
struct Closing {
    double c64;   // value before any fp32 rounding: v (+ w)
    float c32;    // what the reference stores
};
__device__ __forceinline__ Closing closing_value(int d_max, int d_min, int a2, int a_xy, long long sharp, int lam) {
    const double dmax = (double)d_max, dmin = (double)d_min;
    const double r = __ddiv_rn(2.0, dmax);
    const double s = __ddiv_rn(2.0, dmin);
    const double b = __dadd_rn(__dadd_rn(s, r), -2.0);
    const double q = __dadd_rn(__ddiv_rn(1.0, dmin), r);
    const double t = __dmul_rn(q, (double)a2);
    const double v = __fma_rn(t, (double)a_xy, b);
    Closing out;
    out.c64 = v;
    out.c32 = __double2float_rn(v);
    if (lam > 0) {
        const double w = __ddiv_rn((double)sharp, __dmul_rn((double)lam, dmax));
        out.c64 = __dadd_rn(v, w);
        out.c32 = __double2float_rn(__dadd_rn(w, (double)out.c32));
    }
    return out;
}

// The same formula split in two: the part that depends only on (d_max, d_min, A2[x,y], A[x,y]) — the first fp32
// store — and the part that adds sharp/(d_max*lambda) — the second.  closing_finish(closing_first(...), sharp, lam)
// is bit-identical to closing_value(...).c32; candidate scoring computes the first part once per (x,y).
struct ClosingFirst {
    float c32;     // value after the first store
    double dmax;
};
__device__ __forceinline__ ClosingFirst closing_first(int d_max, int d_min, int a2, int a_xy) {
    const double dmax = (double)d_max, dmin = (double)d_min;
    const double r = __ddiv_rn(2.0, dmax);
    const double s = __ddiv_rn(2.0, dmin);
    const double b = __dadd_rn(__dadd_rn(s, r), -2.0);
    const double q = __dadd_rn(__ddiv_rn(1.0, dmin), r);
    const double t = __dmul_rn(q, (double)a2);
    ClosingFirst f;
    f.c32 = __double2float_rn(__fma_rn(t, (double)a_xy, b));
    f.dmax = dmax;
    return f;
}
__device__ __forceinline__ float closing_finish(const ClosingFirst& f, long long sharp, int lam) {
    if (lam <= 0) return f.c32;
    const double w = __ddiv_rn((double)sharp, __dmul_rn((double)lam, f.dmax));
    return __double2float_rn(__dadd_rn(w, (double)f.c32));
}

// The paper-flavour value (bfc_naive.py:31-32 / :39-40) evaluated left to right in fp64 with explicitly rounded
// operations; shared by the paper pass (dcr_bfc_paper.cu) and the paper-flavour SDRF loop (dcr_sdrf.cu).
__device__ __forceinline__ double paper_value(int d1, int d2, int tri, int sq1, int sq2, int gamma) {
    const int dmax = max(d1, d2), dmin = min(d1, d2);
    double t = __ddiv_rn(2.0, (double)d1);
    t = __dadd_rn(t, __ddiv_rn(2.0, (double)d2));
    t = __dadd_rn(t, -2.0);
    t = __dadd_rn(t, __ddiv_rn((double)(2 * (long long)tri), (double)dmax));
    t = __dadd_rn(t, __ddiv_rn((double)tri, (double)dmin));
    if (sq1 > 0 && sq2 > 0) {
        double u = __ddiv_rn(1.0, (double)gamma);
        u = __ddiv_rn(u, (double)dmax);
        u = __dmul_rn(u, (double)(sq1 + sq2));
        t = __dadd_rn(t, u);
    }
    return t;
}

}  // namespace dcr
