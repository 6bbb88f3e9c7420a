// dcr_sdrf.cu — the SDRF rewiring loop as ONE persistent CTA over a device-resident dynamic adjacency.
//
// Takes over the loop body of sdrf_cuda_bfc (rewiring/sdrf_cuda_bfc.py:37-91), utils/softmax.py:4-10 and the
// np.random.choice draw (:64-68).  Per iteration the reference does two dense N^3 matmuls, an N^2 x N kernel,
// two full-matrix arg-reductions with host syncs and one host sync per candidate.  Here an iteration is:
//   1. one scan of the per-entry fp32 curvatures: first-row-major argmin (< 0, else (0,0)) AND argmax (> 0, else
//      (0,0)) of the SAME matrix C_t — the reference's removal step reads the pre-addition C (:39 vs :80);
//   2. candidate scoring (dcr_score.cuh) over (N(x) ∪ {x}) x (N(y) ∪ {y}) in networkx insertion order (:45-54),
//      improvements = fp32(D - C[x,y]) (:59-62);
//   3. the draw: one-hot at the first maximum for tau = inf, else exp(a*tau)/sum and an inverse-CDF look-up with
//      the host-supplied uniform (App. E.3); a uniform within `guard` of a CDF boundary is handed back to the host;
//   4. in-place insertion of (k,l) and removal of the argmax edge in the arena (sorted rows with slack +
//      insertion-order rows), exact support updates;
//   5. incremental refresh of the curvature of the dirty edges only (SURVEY.md App. H): edges at the four touched
//      endpoints and edges closing a triangle with an edge whose support changed.
// No host round trip inside the loop; one 8-int log record per iteration.  The loop is inherently sequential
// (iteration t+1 needs the graph of iteration t), hence one CTA per run; independent runs go side by side, one CTA
// each, in one launch of the batch kernel (dcr_sdrf_run_batch).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <type_traits>
#include <vector>

#include "dcr_directed.cuh"

namespace dcr {

// Loop flavours (template parameter of the loop kernel; loop_kernels() maps DCR_SDRF_MODE_* of dcr.h onto them):
//   LOOP_BFC       sdrf_cuda_bfc, is_undirected=True   (rewiring/sdrf_cuda_bfc.py:14-93) — symmetric arena, maintained
//                  supports, closed-form curvature and scoring (dcr_score.cuh)
//   LOOP_DIRECTED  sdrf_cuda_bfc, is_undirected=False  (:47-49, :72-73, :87-88) — rows [0,n) hold the successors,
//                  rows [n,2n) the predecessors; curvature and scoring by the definition (dcr_directed.cuh)
//   LOOP_CLASSICAL sdrf_no_cuda with '1d' / 'augmented' / 'haantjes' (rewiring/sdrf_no_cuda.py:9-68,
//                  curvature/classical_curvatures.py:6-46) — integer curvatures from the maintained degrees / supports
//   LOOP_PAPER     sdrf_no_cuda's loop with bfc_naive.bfc_edge as the curvature — fp64 paper-flavour values per entry
//                  (paper_eval), scoring in closed form plus one warp per cell of x's row and y's column (DESIGN §4.9)
enum { LOOP_BFC = 0, LOOP_DIRECTED = 1, LOOP_CLASSICAL = 2, LOOP_PAPER = 3 };

#ifndef DCR_SDRF_THREADS
#define DCR_SDRF_THREADS 1024
#endif
constexpr int SDRF_THREADS = DCR_SDRF_THREADS;
constexpr int SDRF_WARPS = SDRF_THREADS / 32;
constexpr uint32_t IMP_MASKED = 0xffffffffu;   // bit pattern marking a masked cell in the improvement matrix
constexpr unsigned long long IMP_MASKED64 = ~0ull;   // (LOOP_PAPER's fp64 cells; a NaN, which no improvement is)
constexpr int STATUS_TOO_MANY_CANDIDATES = DCR_SDRF_TOO_MANY_CANDIDATES;

// Optional phase timers (build with -DDCR_SDRF_PROFILE): cycles per phase summed over the iterations of a launch,
// written to a device array read back with dcr_sdrf_phase_cycles().  Compiled out of the product library.  The array
// is one global without atomics, so only the single-run kernel ticks (TIMED = true); the batch kernel, whose CTAs
// would race on it, instantiates the loop body with TIMED = false.
#ifdef DCR_SDRF_PROFILE
__device__ unsigned long long g_sdrf_phase[16];
#define SDRF_TICK(slot)                                                         \
    do {                                                                        \
        if (TIMED && threadIdx.x == 0) {                                        \
            const long long now__ = clock64();                                  \
            g_sdrf_phase[slot] += (unsigned long long)(now__ - tick__);         \
            tick__ = now__;                                                     \
        }                                                                       \
    } while (0)
#else
#define SDRF_TICK(slot) do { } while (0)
#endif

struct SdrfDev {
    int n;
    int ctype;            // classical loop: 0 = '1d', 1 = 'augmented', 2 = 'haantjes'
    int cap_total;        // arena slots
    int row_cap_max;      // capacity of the per-row scratch arrays
    long long imp_cap;    // cells of the improvement scratch
    int dirty_cap;
    int32_t* rstart;      // [n]
    int32_t* rlen;        // [n]
    int32_t* rcap;        // [n]
    int32_t* selfl;       // [rows] 1: the node lists ITSELF among its neighbours (a self-loop of G that A does not have,
                          //        sdrf_cuda_bfc.py:29 vs :31): one extra entry in the insertion-order row only
    int32_t* col;         // arena: sorted neighbour ids
    int32_t* ord;         // arena: neighbour ids in insertion order (same row offsets)
    int32_t* supp;        // arena: #common neighbours of the entry's edge (A2[i,j])
    float* c32;           // arena: cuda-flavour curvature of the entry
                          // (LOOP_PAPER keeps no supports and no fp32 value: supp / c32 hold the high / low word of the
                          //  entry's fp64 paper-flavour value, so every arena edit moves it unchanged; see paper_get)
    int32_t* owner;       // arena: row id of the slot, -1 = free
    int32_t* flag;        // arena: dedupe flags for the refresh
    int32_t* scalars;     // [0] arena_top, [1] nnz, [2] add edits applied, [3] max_additions (their limit)
    int32_t* base1; int32_t* base2; int32_t* posI; int32_t* posJ;   // score scratch [row_cap_max]
    uint32_t* imp;        // improvement matrix (fp32 bits; LOOP_PAPER: fp64 bits, two words per cell)
    double* pend;         // compact improvements of a pending iteration
    int32_t* dirty;       // pairs (a,b): 2*dirty_cap ints
    int32_t* work;        // slots to refresh: dirty_cap ints
    int32_t* wlist;       // common-neighbour list scratch [row_cap_max]
};

// ------------------------------------------------------------------------------------------------------------
// block-wide primitives (SDRF_THREADS threads, every thread calls)
// ------------------------------------------------------------------------------------------------------------
template <class V>
struct BestT { V v; unsigned long long key; };   // "smaller v wins, then smaller key"
using Best = BestT<float>;                       // (the paper loop compares fp64 values: BestT<double>)

template <class V>
__device__ __forceinline__ BestT<V> best_of(BestT<V> a, BestT<V> b) {
    return (b.v < a.v || (b.v == a.v && b.key < a.key)) ? b : a;
}
template <class V>
__device__ __forceinline__ BestT<V> warp_best(BestT<V> a) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        BestT<V> b;
        b.v = __shfl_xor_sync(FULL, a.v, o);
        b.key = __shfl_xor_sync(FULL, a.key, o);
        a = best_of(a, b);
    }
    return a;
}

struct Reduce {     // shared-memory scratch for the block primitives
    float v[SDRF_WARPS];
    unsigned long long k[SDRF_WARPS];
    double d[SDRF_WARPS];
    long long l[SDRF_WARPS];
    union { Best best; BestT<double> best_d; };
};

template <class V>
__device__ BestT<V> block_best(BestT<V> a, Reduce* r) {
    constexpr bool F64 = sizeof(V) == 8;         // fp64 values go through r->d and r->best_d
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    a = warp_best(a);
    if (lane == 0) {
        if constexpr (F64) r->d[warp] = a.v; else r->v[warp] = a.v;
        r->k[warp] = a.key;
    }
    __syncthreads();
    if (warp == 0) {
        BestT<V> b;
        if constexpr (F64) b.v = lane < SDRF_WARPS ? r->d[lane] : (V)INFINITY;
        else b.v = lane < SDRF_WARPS ? r->v[lane] : INFINITY;
        b.key = lane < SDRF_WARPS ? r->k[lane] : ~0ull;
        b = warp_best(b);
        if (lane == 0) {
            if constexpr (F64) r->best_d = b; else r->best = b;
        }
    }
    __syncthreads();
    BestT<V> out;
    if constexpr (F64) out = r->best_d; else out = r->best;
    __syncthreads();
    return out;
}

// two independent "smaller (v, key) wins" reductions in one go: three barriers instead of six
__device__ void block_best2(Best& a, Best& b, Reduce* r, Reduce* r2) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    a = warp_best(a);
    b = warp_best(b);
    if (lane == 0) { r->v[warp] = a.v; r->k[warp] = a.key; r2->v[warp] = b.v; r2->k[warp] = b.key; }
    __syncthreads();
    if (warp < 2) {
        Reduce* q = warp == 0 ? r : r2;
        Best t;
        t.v = lane < SDRF_WARPS ? q->v[lane] : INFINITY;
        t.key = lane < SDRF_WARPS ? q->k[lane] : ~0ull;
        t = warp_best(t);
        if (lane == 0) q->best = t;
    }
    __syncthreads();
    a = r->best;
    b = r2->best;
    __syncthreads();
}

// exclusive prefix over threads (thread order) + total
__device__ long long block_exscan_ll(long long v, long long* total, Reduce* r) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        long long t = __shfl_up_sync(FULL, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) r->l[warp] = inc;
    __syncthreads();
    long long off = 0, tot = 0;
    for (int w = 0; w < SDRF_WARPS; ++w) {
        if (w < warp) off += r->l[w];
        tot += r->l[w];
    }
    __syncthreads();
    *total = tot;
    return off + inc - v;
}

// exclusive prefixes of a (count, fp64 sum) pair over the threads, plus both totals: one primitive, two barriers
__device__ void block_exscan_pair(long long c, double d, long long* c_off, double* d_off, long long* c_tot,
                                  double* d_tot, Reduce* r) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long ci = c;
    double di = d;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long tc = __shfl_up_sync(FULL, ci, o);
        const double td = __shfl_up_sync(FULL, di, o);
        if (lane >= o) { ci += tc; di = __dadd_rn(di, td); }
    }
    double dex = __shfl_up_sync(FULL, di, 1);
    if (lane == 0) dex = 0.0;
    if (lane == 31) { r->l[warp] = ci; r->d[warp] = di; }
    __syncthreads();
    long long co = 0, ct = 0;
    double dof = 0.0, dt = 0.0;
    for (int w = 0; w < SDRF_WARPS; ++w) {
        if (w < warp) { co += r->l[w]; dof = __dadd_rn(dof, r->d[w]); }
        ct += r->l[w];
        dt = __dadd_rn(dt, r->d[w]);
    }
    __syncthreads();
    *c_off = co + ci - c;
    *d_off = __dadd_rn(dof, dex);
    *c_tot = ct;
    *d_tot = dt;
}

// ------------------------------------------------------------------------------------------------------------
// arena row edits (block-cooperative; arguments are block-uniform)
// ------------------------------------------------------------------------------------------------------------
struct LoopShared {
    Reduce red, red2;
    ScoreShared score;
    int x, y, xr, yr, have_min, have_max;
    float cxy, cmax;
    int n_i, n_j;
    long long n_cand;
    long long chosen_flat;
    long long found_flat;     // first flat index whose CDF exceeds u (atomicMin over the threads)
    int choice, k, l;
    int status, stop, can_add, do_remove;
    double below, above;      // normalised CDF just below / at the chosen candidate
    int cnt_a;                // wlist fill of toggle_supports
    int edit_pos;             // ord_erase: slot of the erased id
};
// the paper loop's extra fields: fp64 extremes and the fields of bfc(x,y) that every interior cell starts from
struct LoopSharedPaper : LoopShared {
    double cxy_d, cmax_d;
    int tri, sq_x, sq_y, gamma;
};

template <class T>
__device__ void shift_left(T* a, int lo, int hi) {    // a[lo-1 .. hi-2] = a[lo .. hi-1]
    for (int base = lo; base < hi; base += SDRF_THREADS) {
        const int idx = base + threadIdx.x;
        T v{};
        const bool on = idx < hi;
        if (on) v = a[idx];
        __syncthreads();
        if (on) a[idx - 1] = v;
        __syncthreads();
    }
}

// the three arrays that follow the SORTED order of a row move together: one pass, two barriers per chunk
__device__ void shift_right3(const SdrfDev& S, int lo, int hi) {
    for (int top = hi; top > lo; top -= SDRF_THREADS) {
        const int base = max(lo, top - SDRF_THREADS);
        const int idx = base + threadIdx.x;
        const bool on = idx < top;
        int32_t c = 0, u = 0;
        float f = 0.0f;
        if (on) { c = S.col[idx]; u = S.supp[idx]; f = S.c32[idx]; }
        __syncthreads();
        if (on) { S.col[idx + 1] = c; S.supp[idx + 1] = u; S.c32[idx + 1] = f; }
        __syncthreads();
    }
}
__device__ void shift_left3(const SdrfDev& S, int lo, int hi) {
    for (int base = lo; base < hi; base += SDRF_THREADS) {
        const int idx = base + threadIdx.x;
        const bool on = idx < hi;
        int32_t c = 0, u = 0;
        float f = 0.0f;
        if (on) { c = S.col[idx]; u = S.supp[idx]; f = S.c32[idx]; }
        __syncthreads();
        if (on) { S.col[idx - 1] = c; S.supp[idx - 1] = u; S.c32[idx - 1] = f; }
        __syncthreads();
    }
}

// make room for one more entry in row v (relocate to the arena top with doubled capacity when full)
__device__ bool row_reserve(const SdrfDev& S, int v) {
    const int len = S.rlen[v], cap = S.rcap[v], start = S.rstart[v], self = S.selfl[v];
    __syncthreads();
    if (len + self < cap) return true;     // (the insertion-order row is `self` entries longer than the sorted one)
    const int ncap = max(2 * cap, 4);
    const int nstart = S.scalars[0];
    if ((long long)nstart + ncap > S.cap_total) return false;
    for (int t = threadIdx.x; t < len + self; t += SDRF_THREADS) {
        S.ord[nstart + t] = S.ord[start + t];
        if (t >= len) continue;
        S.col[nstart + t] = S.col[start + t];
        S.supp[nstart + t] = S.supp[start + t];
        S.c32[nstart + t] = S.c32[start + t];
        S.owner[nstart + t] = v;
        S.owner[start + t] = -1;
        S.c32[start + t] = 0.0f;          // free slots hold 0: the argmin/argmax scan reads values only
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        S.rstart[v] = nstart;
        S.rcap[v] = ncap;
        S.scalars[0] = nstart + ncap;
    }
    __syncthreads();
    return true;
}

// insert `key` into row v (must not be present); new entry gets supp = 0, c32 = 0
__device__ bool row_insert(const SdrfDev& S, int v, int key) {
    if (!row_reserve(S, v)) return false;
    const int start = S.rstart[v], len = S.rlen[v];
    const int pos = start + lower_bound(S.col, start, len, key);
    __syncthreads();
    shift_right3(S, pos, start + len);
    if (threadIdx.x == 0) {
        S.col[pos] = key;
        S.supp[pos] = 0;
        S.c32[pos] = 0.0f;
        S.owner[start + len] = v;
        S.ord[start + len + S.selfl[v]] = key;
        S.rlen[v] = len + 1;
    }
    __syncthreads();
    return true;
}

// erase `key` (must be present) from the insertion-order list S.ord[start .. start+olen)
__device__ void ord_erase(const SdrfDev& S, int start, int olen, int key, LoopShared* sh) {
    if (threadIdx.x == 0) sh->edit_pos = -1;
    __syncthreads();
    for (int t = threadIdx.x; t < olen; t += SDRF_THREADS)
        if (S.ord[start + t] == key) sh->edit_pos = start + t;
    __syncthreads();
    shift_left(S.ord, sh->edit_pos + 1, start + olen);
}

// delete `key` from row v (must be present)
__device__ void row_delete(const SdrfDev& S, int v, int key, LoopShared* sh) {
    const int start = S.rstart[v], len = S.rlen[v];
    const int pos = find_sorted(S.col, start, len, key);
    shift_left3(S, pos + 1, start + len);
    ord_erase(S, start, len + S.selfl[v], key, sh);
    if (threadIdx.x == 0) {
        S.owner[start + len - 1] = -1;
        S.c32[start + len - 1] = 0.0f;    // free slots hold 0
        S.rlen[v] = len - 1;
    }
    __syncthreads();
}

// LOOP_PAPER: the fp64 value of the entry at `slot`, stored as its high word in supp and its low word in c32 (bit moves
// only: nothing does float arithmetic on those words in this loop); a free or new slot reads +0.0
__device__ __forceinline__ double paper_get(const SdrfDev& S, int slot) {
    return __hiloint2double(S.supp[slot], __float_as_int(S.c32[slot]));
}
__device__ __forceinline__ void paper_put(const SdrfDev& S, int slot, double v) {
    S.supp[slot] = __double2hiint(v);
    S.c32[slot] = __int_as_float(__double2loint(v));
}

// append the entry (a,b) to the dirty list; undirected callers pass (min, max) so an edge always names one slot
__device__ __forceinline__ void push_dirty(const SdrfDev& S, int* counter, int a, int b) {
    const int p = atomicAdd(counter, 1);
    if (p < S.dirty_cap) {
        S.dirty[2 * p] = a;
        S.dirty[2 * p + 1] = b;
    }
}

// Exact support update + dirty marking for toggling edge (k,l); the edge must currently be PRESENT in the arena.
// delta = +1 after an insertion, -1 before a deletion.
template <bool CLOSING_EDGES>
__device__ void toggle_supports(const SdrfDev& S, const GraphView& g, int k, int l, int delta, int* dirty_count,
                                LoopShared* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sk = S.rstart[k], dk = S.rlen[k], sl = S.rstart[l], dl = S.rlen[l];
    if (threadIdx.x == 0) sh->cnt_a = 0;
    __syncthreads();
    // every edge at k and at l is dirty (degree change)
    for (int t = threadIdx.x; t < dk; t += SDRF_THREADS) {
        const int w = S.col[sk + t];
        push_dirty(S, dirty_count, min(k, w), max(k, w));
    }
    for (int t = threadIdx.x; t < dl; t += SDRF_THREADS) {
        const int w = S.col[sl + t];
        push_dirty(S, dirty_count, min(l, w), max(l, w));
    }
    // W = N(k) ∩ N(l): four support entries per common neighbour change by delta
    for (int t = threadIdx.x; t < dk; t += SDRF_THREADS) {
        const int w = S.col[sk + t];
        const int q = find_sorted(S.col, sl, dl, w);
        if (q >= 0) {
            S.supp[sk + t] += delta;
            S.supp[q] += delta;
            S.supp[edge_slot(g, w, k)] += delta;
            S.supp[edge_slot(g, w, l)] += delta;
            S.wlist[atomicAdd(&sh->cnt_a, 1)] = w;
        }
    }
    __syncthreads();
    const int nw = sh->cnt_a;
    if (threadIdx.x == 0 && delta > 0) {
        S.supp[edge_slot(g, k, l)] = nw;
        S.supp[edge_slot(g, l, k)] = nw;
    }
    // edges (w,z) closing a triangle with (k,w) or (l,w): their "support == 1" counts may change (BFC only; the
    // classical curvatures read nothing but the degrees and the support of the edge itself)
    for (int t = warp; CLOSING_EDGES && t < nw; t += SDRF_WARPS) {
        const int w = S.wlist[t];
        const int sw = S.rstart[w], dw = S.rlen[w];
        for (int p = lane; p < dw; p += 32) {
            const int z = S.col[sw + p];
            if (z == k || z == l) continue;
            if (find_sorted(S.col, sk, dk, z) >= 0 || find_sorted(S.col, sl, dl, z) >= 0)
                push_dirty(S, dirty_count, min(w, z), max(w, z));
        }
    }
    __syncthreads();
}

// cuda-flavour curvature of the entry at `slot` from the maintained supports (warp-cooperative)
__device__ __forceinline__ float entry_curvature(const SdrfDev& S, int a, int b, int slot_ab, int lane) {
    int sa = S.rstart[a], da = S.rlen[a], sb = S.rstart[b], db = S.rlen[b];
    const int dmax = max(da, db), dmin = min(da, db), di_dj = da + db;
    if (da > db) { int t = da; da = db; db = t; t = sa; sa = sb; sb = t; }
    int ta = 0, tb = 0;
    for (int t = lane; t < da; t += 32) {
        const int q = find_sorted(S.col, sb, db, S.col[sa + t]);
        if (q >= 0) { ta += S.supp[sa + t] == 1; tb += S.supp[q] == 1; }
    }
    ta = warp_sum(ta);
    tb = warp_sum(tb);
    return closing_value(dmax, dmin, S.supp[slot_ab], 1, di_dj - ta - tb, dmax).c32;
}

// classical curvature of an entry from the maintained degrees / support (curvature/classical_curvatures.py:15-28);
// small integers, exact in fp32
__device__ __forceinline__ float classical_curvature(const SdrfDev& S, int a, int b, int slot_ab) {
    // a self-loop of G counts twice in G.degree and makes the node its own neighbour: for an EDGE (a,b) each looped
    // endpoint is one more common neighbour (a in N(b) and in N'(a) = N(a) + {a})
    const int la = S.selfl[a], lb = S.selfl[b];
    const int base = 4 - (S.rlen[a] + 2 * la) - (S.rlen[b] + 2 * lb);
    const int tri = S.supp[slot_ab] + la + lb;
    if (S.ctype == 0) return (float)base;                 // '1d'
    if (S.ctype == 1) return (float)(base + 3 * tri);      // 'augmented'
    return (float)tri;                                    // 'haantjes'
}
// curvature of the loop edge (u,u) itself (compute_curvature_edge with v1 = v2 = u): degree d + 2, N'(u) ∩ N'(u) = d + 1
__device__ __forceinline__ float classical_loop_curvature(const SdrfDev& S, int u) {
    const int d = S.rlen[u];
    if (S.ctype == 0) return (float)(4 - 2 * (d + 2));
    if (S.ctype == 1) return (float)(4 - 2 * (d + 2) + 3 * (d + 1));
    return (float)(d + 1);
}

// Directed loop: entries whose curvature may change when the entry k -> l is toggled (call while it is PRESENT).
// C[i,j] reads d_in[i], d_out[j], N_out(i), N_in(j), A2[i,*] over N_in(j) and A2[*,j] over N_out(i)
// (bfc_cuda.py:20-44); A2[a,b] changes iff (a = k and l -> b) or (b = l and a -> k).  Hence: the entries leaving k
// and l, the entries arriving at k and l, and the entries i -> j with i -> k and l -> j.
__device__ void directed_mark_dirty(const SdrfDev& S, int k, int l, int* dirty_count) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = S.n;
    const int sok = S.rstart[k], nok = S.rlen[k], sol = S.rstart[l], nol = S.rlen[l];
    const int sik = S.rstart[n + k], nik = S.rlen[n + k], sil = S.rstart[n + l], nil = S.rlen[n + l];
    for (int t = threadIdx.x; t < nok; t += SDRF_THREADS) push_dirty(S, dirty_count, k, S.col[sok + t]);
    for (int t = threadIdx.x; t < nol; t += SDRF_THREADS) push_dirty(S, dirty_count, l, S.col[sol + t]);
    for (int t = threadIdx.x; t < nik; t += SDRF_THREADS) push_dirty(S, dirty_count, S.col[sik + t], k);
    for (int t = threadIdx.x; t < nil; t += SDRF_THREADS) push_dirty(S, dirty_count, S.col[sil + t], l);
    for (int t = warp; t < nik; t += SDRF_WARPS) {
        const int i = S.col[sik + t];
        const int soi = S.rstart[i], noi = S.rlen[i];
        for (int p = lane; p < noi; p += 32) {
            const int j = S.col[soi + p];
            if (find_sorted(S.col, sol, nol, j) >= 0) push_dirty(S, dirty_count, i, j);
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------------------
// paper loop: bfc_naive.bfc_edge over the arena's sorted rows (DESIGN §4.9)
// ------------------------------------------------------------------------------------------------------------
// The arena graph plus at most one VIRTUAL edge {p,q} that is not in it (p = q = -1: none): candidate scoring
// evaluates bfc(x,y) on G + (i,j) without editing the arena.
struct PaperView {
    GraphView g;
    int p, q;
    __device__ __forceinline__ int deg(int a) const { return g.degree(a) + (a == p || a == q); }
    // t-th neighbour of a: the sorted row, then the virtual neighbour
    __device__ __forceinline__ int nb(int a, int t) const {
        return t < g.degree(a) ? g.col[g.begin(a) + t] : (a == p ? q : p);
    }
    __device__ __forceinline__ bool has(int a, int b) const {
        return (a == p && b == q) || (a == q && b == p) || find_sorted(g.col, g.begin(a), g.degree(a), b) >= 0;
    }
};

// For the edge (a,b) and k in N(a): c(k) = |N(k) ∩ M_b| with M_b = N(b) \ N(a) \ {a} when k is in M_a (then k is a
// square at a iff c(k) > 0, and bfc_naive.py:36-37 gives gamma = max c(k)); -1 when k = b or k is a common
// neighbour (a triangle).  Serial over the shorter of N(k) and N(b).
__device__ __forceinline__ int paper_c(const PaperView& v, int a, int b, int k) {
    if (k == b || v.has(b, k)) return -1;
    const int dk = v.deg(k), db = v.deg(b);
    int c = 0;
    if (dk <= db) {
        for (int s = 0; s < dk; ++s) {
            const int w = v.nb(k, s);
            c += w != a && v.has(b, w) && !v.has(a, w);
        }
    } else {
        for (int s = 0; s < db; ++s) {
            const int w = v.nb(b, s);
            c += w != a && !v.has(a, w) && v.has(k, w);
        }
    }
    return c;
}

// bfc_naive.bfc_edge(G, u, v) of the edge (u,v) (warp-cooperative, every lane returns it): the int 0 of :18-19 when
// deg_min == 1, else paper_value over tri, |□_u|, |□_v| and gamma — bit-identical to the paper pass.
__device__ double paper_eval(const PaperView& v, int u, int w, int lane) {
    const int du = v.deg(u), dw = v.deg(w);
    if (min(du, dw) <= 1) return 0.0;
    int tri = 0, sq_u = 0, sq_w = 0, gam = 0;
    for (int t = lane; t < du; t += 32) {
        const int k = v.nb(u, t);
        const int c = paper_c(v, u, w, k);
        tri += c < 0 && k != w;
        sq_u += c > 0;
        gam = max(gam, c);
    }
    for (int t = lane; t < dw; t += 32) {
        const int c = paper_c(v, w, u, v.nb(w, t));
        sq_w += c > 0;
        gam = max(gam, c);
    }
    return paper_value(du, dw, warp_sum(tri), warp_sum(sq_u), warp_sum(sq_w), warp_max(gam));
}

// Paper loop: edges whose bfc_edge may change when {k,l} is toggled (call with the edge present).  For an edge (u,v)
// away from k and l, N(u), N(v), tri and M_u, M_v stay; only c(k) or c(l) can change, and only when k is in M_u and
// l in M_v (or mirrored).  Hence: the edges at k and at l, and the edges (a,b) with a in N(k), b in N(l).  Each
// directed entry is pushed at most once by the second part: at most 2 nnz pairs per toggle.
__device__ void paper_mark_dirty(const SdrfDev& S, int k, int l, int* dirty_count) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sk = S.rstart[k], dk = S.rlen[k], sl = S.rstart[l], dl = S.rlen[l];
    for (int t = threadIdx.x; t < dk; t += SDRF_THREADS) {
        const int w = S.col[sk + t];
        push_dirty(S, dirty_count, min(k, w), max(k, w));
    }
    for (int t = threadIdx.x; t < dl; t += SDRF_THREADS) {
        const int w = S.col[sl + t];
        push_dirty(S, dirty_count, min(l, w), max(l, w));
    }
    for (int t = warp; t < dk; t += SDRF_WARPS) {
        const int a = S.col[sk + t];
        if (a == l) continue;                                  // (its edges are at l)
        const int sa = S.rstart[a], da = S.rlen[a];
        for (int p = lane; p < da; p += 32) {
            const int b = S.col[sa + p];
            if (b != k && find_sorted(S.col, sl, dl, b) >= 0) push_dirty(S, dirty_count, min(a, b), max(a, b));
        }
    }
    __syncthreads();
}

// Paper loop: improvements bfc(x,y) on G + (i,j) minus bfc(x,y) on G for every cell, fp64 bits into imp64 (masked
// cells as the other loops).  With c(k) of (x,y) computed once (base1 over N(x), base2 over N(y)):
//   i in M_x, j in M_y : degrees and tri stay, c(i) and c(j) grow by one, nothing else moves —
//                        |□_x| += [c(i) = 0], |□_y| += [c(j) = 0], gamma = max(gamma, c(i) + 1, c(j) + 1);
//   i or j a common neighbour : nothing bfc(x,y) reads changes, improvement 0;
//   i = x (row n_i - 1) or j = y (column n_j - 1) : one warp per cell, paper_eval with the virtual edge (i,j).
template <class NbI, class NbJ>
__device__ void paper_score(const SdrfDev& S, const GraphView& g, int x, int y, NbI nbI, int n_i, NbJ nbJ, int n_j,
                            double cxy, unsigned long long* imp64, LoopSharedPaper* sh) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const PaperView none{g, -1, -1};
    const int mi = n_i - 1, mj = n_j - 1;              // x's and y's neighbours (x and y themselves come last)
    if (tid == 0) { sh->tri = 0; sh->sq_x = 0; sh->sq_y = 0; sh->gamma = 0; }
    __syncthreads();
    for (int t = tid; t < mi + mj; t += SDRF_THREADS) {
        const bool ys = t >= mi;
        const int c = ys ? paper_c(none, y, x, nbJ(t - mi)) : paper_c(none, x, y, nbI(t));
        (ys ? S.base2 : S.base1)[ys ? t - mi : t] = c;
        if (c > 0) {
            atomicAdd(ys ? &sh->sq_y : &sh->sq_x, 1);
            atomicMax(&sh->gamma, c);
        }
        if (!ys && c < 0 && nbI(t) != y) atomicAdd(&sh->tri, 1);
    }
    __syncthreads();
    const int dx = S.rlen[x], dy = S.rlen[y];
    const int tri = sh->tri, sq_x = sh->sq_x, sq_y = sh->sq_y, gam = sh->gamma;
    const long long cells = (long long)n_i * n_j;
    for (long long c = tid; c < cells; c += SDRF_THREADS) {
        const int I = (int)(c / n_j), J = (int)(c - (long long)I * n_j);
        const int i = nbI(I), j = nbJ(J);
        if (i == j || edge_slot(g, i, j) >= 0) { imp64[c] = IMP_MASKED64; continue; }
        if (I == mi || J == mj) continue;                                // the warp pass below
        const int ci = S.base1[I], cj = S.base2[J];
        double d = 0.0;
        if (ci >= 0 && cj >= 0) {
            const double after = min(dx, dy) <= 1 ? 0.0
                                 : paper_value(dx, dy, tri, sq_x + (ci == 0), sq_y + (cj == 0),
                                               max(gam, max(ci, cj) + 1));
            d = __dsub_rn(after, cxy);
        }
        imp64[c] = (unsigned long long)__double_as_longlong(d);
    }
    for (int t = warp; t < mi + mj; t += SDRF_WARPS) {
        const bool row = t < mj;
        const int I = row ? mi : t - mj, J = row ? t : mj;
        const int i = nbI(I), j = nbJ(J);
        if (i == j || edge_slot(g, i, j) >= 0) continue;
        const double after = paper_eval(PaperView{g, i, j}, x, y, lane);
        if (lane == 0) imp64[(long long)I * n_j + J] = (unsigned long long)__double_as_longlong(__dsub_rn(after, cxy));
    }
}

// ------------------------------------------------------------------------------------------------------------
// initialisation kernels over arena slots (multi-CTA)
// ------------------------------------------------------------------------------------------------------------
// One warp per arena slot s.  The single-state kernels and the batched ones of dcr_sdrf_create_batch call the same
// per-entry bodies, so a value is computed by the same code on either path.
__device__ __forceinline__ void init_support_entry(const SdrfDev& S, int s, int lane) {
    const int a = S.owner[s];
    if (a < 0) return;
    const int c = warp_intersect_count(GraphView{S.rstart, S.rlen, S.col}, a, S.col[s], lane);
    if (lane == 0) S.supp[s] = c;
}
template <int MODE>
__device__ __forceinline__ void init_curvature_entry(const SdrfDev& S, int s, int lane) {
    const int a = S.owner[s];
    if (a < 0) return;
    if constexpr (MODE == LOOP_PAPER) {
        const double c = paper_eval(PaperView{{S.rstart, S.rlen, S.col}, -1, -1}, a, S.col[s], lane);
        if (lane == 0) paper_put(S, s, c);
        return;
    }
    float c;
    if constexpr (MODE == LOOP_DIRECTED) {
        if (a >= S.n) return;                   // predecessor rows carry no curvature
        const GraphView gout{S.rstart, S.rlen, S.col}, gin{S.rstart + S.n, S.rlen + S.n, S.col};
        c = directed_entry_curvature(gout, gin, a, S.col[s], lane).c32;
    } else if constexpr (MODE == LOOP_CLASSICAL) {
        c = classical_curvature(S, a, S.col[s], s);
    } else {
        c = entry_curvature(S, a, S.col[s], s, lane);
    }
    if (lane == 0) S.c32[s] = c;
}
__global__ void sdrf_init_support_kernel(SdrfDev S, int top) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; s < top; s += warps) init_support_entry(S, s, lane);
}
template <int MODE>
__global__ void sdrf_init_curvature_kernel(SdrfDev S, int top) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; s < top; s += warps) init_curvature_entry<MODE>(S, s, lane);
}

// ------------------------------------------------------------------------------------------------------------
// set-up of many states in one pass (dcr_sdrf_create_batch)
// ------------------------------------------------------------------------------------------------------------
// Per-state record of the batched set-up; `stage` points at the state's part of the packed staging buffer:
// rstart, rlen, rcap, selfl [rows each], col, ord, owner [used each], scalars [8], all int32.
struct SdrfInitDesc {
    SdrfDev S;
    const int32_t* stage;
    int rows, used;       // used: arena slots filled at set-up (sum of the row capacities)
};
static_assert(sizeof(SdrfInitDesc) % 8 == 0, "descriptor table packed as 8-byte words");

// the state whose range [off[b], off[b+1]) holds t (off: count+1 non-decreasing offsets, off[0] = 0 <= t < off[count])
__device__ __forceinline__ int state_of(const long long* __restrict__ off, int count, long long t) {
    int lo = 0, hi = count - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= t) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// Fills every state's persistent arrays from the staging buffer and clears the rest of its arena, as
// sdrf_create_impl's copies and memsets do: unit t of state b is arena slot t (t < cap_total) or row t - cap_total.
// off[b] = sum over earlier states of cap_total + rows.
__global__ void sdrf_batch_setup_kernel(const SdrfInitDesc* __restrict__ descs, const long long* __restrict__ off,
                                        int count) {
    const long long total = off[count];
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int b = state_of(off, count, t);
        const SdrfInitDesc& d = descs[b];
        const SdrfDev& S = d.S;
        const long long i = t - off[b];
        const int32_t* st = d.stage;
        if (i < S.cap_total) {
            const int s = (int)i;
            const int32_t* cols = st + 4 * d.rows;
            if (s < d.used) {
                S.col[s] = cols[s];
                S.ord[s] = cols[d.used + s];
            }
            S.owner[s] = s < d.used ? cols[2 * d.used + s] : -1;
            S.flag[s] = 0;
            S.supp[s] = 0;
            S.c32[s] = 0.0f;
            if (s < 8) S.scalars[s] = cols[3 * d.used + s];
        } else {
            const int r = (int)(i - S.cap_total);
            S.rstart[r] = st[r];
            S.rlen[r] = st[d.rows + r];
            S.rcap[r] = st[2 * d.rows + r];
            S.selfl[r] = st[3 * d.rows + r];
        }
    }
}
// one warp per filled arena slot of every state (off[b] = sum over earlier states of `used`)
__global__ void sdrf_batch_init_support_kernel(const SdrfInitDesc* __restrict__ descs, const long long* __restrict__ off,
                                               int count) {
    const int lane = threadIdx.x & 31;
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; w < off[count]; w += warps) {
        const int b = state_of(off, count, w);
        init_support_entry(descs[b].S, (int)(w - off[b]), lane);
    }
}
template <int MODE>
__global__ void sdrf_batch_init_curvature_kernel(const SdrfInitDesc* __restrict__ descs,
                                                 const long long* __restrict__ off, int count) {
    const int lane = threadIdx.x & 31;
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; w < off[count]; w += warps) {
        const int b = state_of(off, count, w);
        init_curvature_entry<MODE>(descs[b].S, (int)(w - off[b]), lane);
    }
}

__device__ __forceinline__ float val_min(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ float val_max(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double val_min(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ double val_max(double a, double b) { return fmax(a, b); }

// ------------------------------------------------------------------------------------------------------------
// one edge toggle, shared by the loop (step 4 / 5) and the edit kernel
// ------------------------------------------------------------------------------------------------------------
// G.add_edge(k, l) on the arena (the edge must be absent): both rows append in insertion order (directed: the
// successor row of k and the predecessor row of l); false when the arena is full
template <int MODE>
__device__ __forceinline__ bool edge_insert(const SdrfDev& S, int k, int l) {
    constexpr int L_ROW = (MODE == LOOP_DIRECTED);  // directed: the mirror entry lives in the predecessor rows
    bool ok = row_insert(S, k, l);
    ok = ok && row_insert(S, L_ROW * S.n + l, k);
    if (!ok) return false;
    if (threadIdx.x == 0) S.scalars[1] += L_ROW ? 1 : 2;
    __syncthreads();
    return true;
}
// G.remove_edge(k, l) on the arena (the edge must be present)
template <int MODE>
__device__ __forceinline__ void edge_delete(const SdrfDev& S, int k, int l, LoopShared* sh) {
    constexpr int L_ROW = (MODE == LOOP_DIRECTED);
    row_delete(S, k, l, sh);
    row_delete(S, L_ROW * S.n + l, k, sh);
    if (threadIdx.x == 0) S.scalars[1] -= L_ROW ? 1 : 2;
    __syncthreads();
}
// the flavour's support update and dirty rule for toggling {k,l}; call while the edge is PRESENT (after the insertion,
// before the deletion); delta = +1 for an insertion, -1 for a deletion
template <int MODE>
__device__ __forceinline__ void toggle_mark(const SdrfDev& S, const GraphView& g, int k, int l, int delta,
                                            int* dirty_count, LoopShared* sh) {
    if constexpr (MODE == LOOP_DIRECTED) directed_mark_dirty(S, k, l, dirty_count);
    else if constexpr (MODE == LOOP_PAPER) paper_mark_dirty(S, k, l, dirty_count);
    else toggle_supports<MODE == LOOP_BFC>(S, g, k, l, delta, dirty_count, sh);
}
// Refresh the curvature of the first nd dirty pairs (nd <= dirty_cap): dedupe them into slots (S.work, counted in
// *work_count, which the caller zeroed) and re-evaluate each slot once, one warp per slot.
template <int MODE>
__device__ __forceinline__ void refresh_dirty(const SdrfDev& S, const GraphView& g, const GraphView& gin, int nd,
                                              int* work_count) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int t = tid; t < nd; t += SDRF_THREADS) {
        const int a = S.dirty[2 * t], b = S.dirty[2 * t + 1];
        const int s = edge_slot(g, a, b);
        if (s >= 0 && atomicExch(&S.flag[s], 1) == 0) S.work[atomicAdd(work_count, 1)] = s;
    }
    __syncthreads();
    const int nwk = *work_count;
    for (int t = warp; t < nwk; t += SDRF_WARPS) {
        const int s = S.work[t];
        const int a = S.owner[s], b = S.col[s];
        if constexpr (MODE == LOOP_PAPER) {
            const double c = paper_eval(PaperView{g, -1, -1}, a, b, lane);
            if (lane == 0) {
                paper_put(S, s, c);
                paper_put(S, edge_slot(g, b, a), c);
                S.flag[s] = 0;
            }
            continue;
        }
        float c;
        if constexpr (MODE == LOOP_DIRECTED) c = directed_entry_curvature(g, gin, a, b, lane).c32;
        else if constexpr (MODE == LOOP_CLASSICAL) c = classical_curvature(S, a, b, s);
        else c = entry_curvature(S, a, b, s, lane);
        if (lane == 0) {
            S.c32[s] = c;
            if (MODE != LOOP_DIRECTED) S.c32[edge_slot(g, b, a)] = c;   // symmetric A: C[b,a] == C[a,b] bit for bit
            S.flag[s] = 0;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// candidate scoring of one pair (x, y), shared by the loop (step 2) and sdrf_score_kernel
// ------------------------------------------------------------------------------------------------------------
// The candidate list of one side in networkx order (sdrf_cuda_bfc.py:45-49): the insertion-order row of `row` (x's
// neighbours / successors, y's neighbours / predecessors; a node that lists itself appears in it) and then the node
// itself.  n = row length + self entry + 1.
struct CandList {
    const int32_t* ord;
    int o, n, self;
    __device__ __forceinline__ int operator()(int t) const { return t < n - 1 ? ord[o + t] : self; }
};
__device__ __forceinline__ int cand_count(const SdrfDev& S, int row) { return S.rlen[row] + S.selfl[row] + 1; }

// Scores every cell (I, J) of nbI x nbJ for the pair (x, y).  BFC / directed: put(I, J, D) with D the curvature of
// (x, y) after adding (i, j), MASKED_D for a masked cell; classical: put(I, J, improvement) in closed form, MASKED_D
// for a masked cell; paper: the fp64 bits of the improvement (IMP_MASKED64 when masked) into imp64[I * n_j + J],
// against cxy_d = bfc(x, y).  Reads the state and writes only its scratch rows (sc; the paper flavour: S.base1 / base2),
// imp64 / put and the shared structs.  Every thread calls.
// after_prepare() runs between the BFC flavour's two scoring phases (the loop's phase timer).
template <int MODE, class Put, class Sh, class Hook>
__device__ __forceinline__ void score_pair(const SdrfDev& S, const GraphView& g, const GraphView& gin, int x, int y,
                                           const CandList& nbI, const CandList& nbJ, const ScoreScratch& sc, Put put,
                                           unsigned long long* imp64, double cxy_d, Sh* sh, DirScoreShared* dsh,
                                           int* dred, Hook after_prepare) {
    const int n_i = nbI.n, n_j = nbJ.n;
    if constexpr (MODE == LOOP_BFC) {
        score_prepare(g, S.supp, x, y, nbI, n_i, nbJ, n_j, sc, &sh->score);
        after_prepare();
        // x (y) sits at the end of its list — and, with a self-loop, once more inside it: then every row is checked
        score_cells(g, S.supp, x, y, nbI, n_i, nbJ, n_j, sc, &sh->score, put, S.selfl[x] ? -1 : n_i - 1,
                    S.selfl[y] ? -1 : n_j - 1);
    } else if constexpr (MODE == LOOP_DIRECTED) {
        directed_score_prepare(g, gin, x, y, nbI, n_i, nbJ, n_j, sc, dsh, dred);
        directed_score_cells(g, gin, x, y, nbI, n_i, nbJ, n_j, sc, dsh, put);
    } else if constexpr (MODE == LOOP_PAPER) {
        paper_score(S, g, x, y, nbI, n_i, nbJ, n_j, cxy_d, imp64, sh);
    } else {
        // sdrf_no_cuda.py:41-46 in closed form: adding (i,j) changes curvature(x,y) only when it touches x or y.
        // i == x (then j in N(y)\N(x)): deg x + 1 and one more triangle; j == y mirrored; every other
        // candidate leaves both degrees and the common neighbours alone.
        const float special = S.ctype == 0 ? -1.0f : (S.ctype == 1 ? 2.0f : 1.0f);
        const long long cells = (long long)n_i * n_j;
        for (long long c = threadIdx.x; c < cells; c += SDRF_THREADS) {
            const int I = (int)(c / n_j), J = (int)(c - (long long)I * n_j);
            const int i = nbI(I), j = nbJ(J);
            const bool masked = (i == j) || edge_slot(g, i, j) >= 0;       // :34
            put(I, J, masked ? MASKED_D : ((i == x || j == y) ? special : 0.0f));
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// the loop
// ------------------------------------------------------------------------------------------------------------
// One run of the loop on the calling CTA.  Block-uniform arguments only; nothing here reads blockIdx or gridDim, so the
// single-run kernel and every CTA of the batch kernel execute the same code on their own state.
template <int MODE, bool TIMED>
__device__ __forceinline__ void sdrf_loop_body(const SdrfDev& S, int loops, int remove_edges, float bound32,
                                               double bound64, double tau, int tau_inf,
                                               const double* __restrict__ uniforms, long long n_uniforms,
                                               int forced_choice, double guard, int32_t* __restrict__ log,
                                               dcr_sdrf_result* __restrict__ result) {
    constexpr bool PAPER = MODE == LOOP_PAPER;
    constexpr bool NX_LOOP = MODE == LOOP_CLASSICAL || PAPER;     // sdrf_no_cuda's loop: min / max over G.edges
    using Val = std::conditional_t<PAPER, double, float>;         // entry values, extremes and improvements
    using Bits = std::conditional_t<PAPER, unsigned long long, uint32_t>;   // improvement matrix cells
    constexpr Bits MASKED = PAPER ? IMP_MASKED64 : IMP_MASKED;
    auto imp_at = [&](long long f) -> Bits { return reinterpret_cast<const Bits*>(S.imp)[f]; };
    auto value = [&](int s) -> Val {
        if constexpr (PAPER) return paper_get(S, s); else return S.c32[s];
    };
    auto imp_val = [](Bits b) -> Val {
        if constexpr (PAPER) return __longlong_as_double((long long)b); else return __uint_as_float(b);
    };
    __shared__ std::conditional_t<PAPER, LoopSharedPaper, LoopShared> sh;
    __shared__ DirScoreShared dsh;
    __shared__ int dirty_count, work_count, dred[2];
    const int tid = threadIdx.x;
    GraphView g{S.rstart, S.rlen, S.col};                       // undirected adjacency / successors
    GraphView gin{S.rstart + S.n, S.rlen + S.n, S.col};         // predecessors (directed loop only)
    ScoreScratch sc{S.base1, S.base2, S.posI, S.posJ};
    int it = 0, draws = 0;
    if (tid == 0) { sh.status = DCR_SDRF_OK; sh.stop = 0; }
    __syncthreads();

#ifdef DCR_SDRF_PROFILE
    long long tick__ = clock64();
#endif
    for (; it < loops; ++it) {
        const int top = S.scalars[0];
        if constexpr (NX_LOOP) {
            // ---- 1c. min(G.edges, key=curvature) / max(...) (sdrf_no_cuda.py:27, :59-61) --------------------
            // G.edges lists every edge once, from its first endpoint in node order, neighbours in insertion order:
            // the first minimum is at the smallest u that has an entry (u, v > u) with the minimal value, and among
            // those at the earliest position of u's insertion-order row.  The maximum is taken over the same C_t
            // (curv_dict predates the addition; the new edge is excluded, :59).
            Val vmin = INFINITY, vmax = -INFINITY;
            for (int s = tid; s < top; s += SDRF_THREADS) {
                if (S.owner[s] < 0) continue;
                const Val v = value(s);
                vmin = val_min(vmin, v);
                vmax = val_max(vmax, v);
            }
            for (int u = tid; !PAPER && u < S.n; u += SDRF_THREADS) {     // the loop edges (u,u) of G.edges
                if (!S.selfl[u]) continue;
                const float v = classical_loop_curvature(S, u);
                vmin = fminf(vmin, v);
                vmax = fmaxf(vmax, v);
            }
            vmin = block_best(BestT<Val>{vmin, 0ull}, &sh.red).v;
            vmax = -block_best(BestT<Val>{-vmax, 0ull}, &sh.red).v;
            if (!(vmin <= vmax)) {                              // no edges: min() of an empty sequence
                if (tid == 0) sh.status = DCR_SDRF_EMPTY_GRAPH;
                __syncthreads();
                break;
            }
            unsigned long long umin = ~0ull, umax = ~0ull;
            for (int s = tid; s < top; s += SDRF_THREADS) {
                const int o = S.owner[s];
                if (o < 0 || S.col[s] < o) continue;
                const Val v = value(s);
                if (v == vmin) umin = min(umin, (unsigned long long)o);
                if (v == vmax) umax = min(umax, (unsigned long long)o);
            }
            for (int u = tid; !PAPER && u < S.n; u += SDRF_THREADS) {
                if (!S.selfl[u]) continue;
                const float v = classical_loop_curvature(S, u);
                if (v == vmin) umin = min(umin, (unsigned long long)u);
                if (v == vmax) umax = min(umax, (unsigned long long)u);
            }
            const int xu = (int)block_best(Best{0.0f, umin}, &sh.red).key;
            const int xru = (int)block_best(Best{0.0f, umax}, &sh.red).key;
            // this thread's first position in u's insertion-order row of an entry (u, v >= u) of value `val` (the row
            // holds the node itself where its loop was added: G.edges reports it there)
            auto first_pos = [&](int u, Val val) {
                const int st = S.rstart[u], len = S.rlen[u];
                unsigned long long p = ~0ull;
                for (int t = tid; t < len + S.selfl[u]; t += SDRF_THREADS) {
                    const int v = S.ord[st + t];
                    const bool hit = v == u ? classical_loop_curvature(S, u) == val
                                            : (v > u && value(find_sorted(S.col, st, len, v)) == val);
                    if (hit) p = min(p, (unsigned long long)t);
                }
                return p;
            };
            unsigned long long pmin = first_pos(xu, vmin), pmax = first_pos(xru, vmax);
            pmin = block_best(Best{0.0f, pmin}, &sh.red).key;
            pmax = block_best(Best{0.0f, pmax}, &sh.red).key;
            if (tid == 0) {
                sh.have_min = 1; sh.have_max = 1;
                sh.x = xu;  sh.y = S.ord[S.rstart[xu] + (int)pmin];
                sh.xr = xru; sh.yr = S.ord[S.rstart[xru] + (int)pmax];
                if constexpr (PAPER) { sh.cxy_d = vmin; sh.cmax_d = vmax; }
                else { sh.cxy = vmin; sh.cmax = vmax; }
            }
        } else {
        // ---- 1. argmin / argmax of C_t (sdrf_cuda_bfc.py:40-42, :80-82) ---------------------------------
        // Pass 1 reads only the curvatures (free slots hold 0, which is neither < 0 nor > 0) and reduces the two
        // extreme VALUES; pass 2 visits the few slots that attain them and reduces the first row-major key.
        // (Directed loop: predecessor rows keep c32 = 0, so only successor entries can attain an extreme.)
        // One pass: every thread keeps its best (value, first row-major key) for the minimum and for the maximum (the
        // key is only fetched when a slot improves or ties the thread's current best), then ONE fused block reduction.
        Best bmin{0.0f, ~0ull}, bmax{0.0f, ~0ull};   // bmax holds the NEGATED value
        for (int s = tid; s < top; s += SDRF_THREADS) {
            const float v = S.c32[s];
            if (v < 0.0f && v <= bmin.v) {
                const unsigned long long key = ((unsigned long long)(unsigned)S.owner[s] << 32) | (unsigned)S.col[s];
                if (v < bmin.v || key < bmin.key) { bmin.v = v; bmin.key = key; }
            }
            if (v > 0.0f && -v <= bmax.v) {
                const unsigned long long key = ((unsigned long long)(unsigned)S.owner[s] << 32) | (unsigned)S.col[s];
                if (-v < bmax.v || key < bmax.key) { bmax.v = -v; bmax.key = key; }
            }
        }
        block_best2(bmin, bmax, &sh.red, &sh.red2);
        if (tid == 0) {
            sh.have_min = bmin.v < 0.0f;
            sh.x = sh.have_min ? (int)(bmin.key >> 32) : 0;
            sh.y = sh.have_min ? (int)(bmin.key & 0xffffffffu) : 0;
            sh.cxy = sh.have_min ? bmin.v : 0.0f;
            sh.have_max = bmax.v < 0.0f;
            sh.xr = sh.have_max ? (int)(bmax.key >> 32) : 0;
            sh.yr = sh.have_max ? (int)(bmax.key & 0xffffffffu) : 0;
            sh.cmax = sh.have_max ? -bmax.v : 0.0f;
        }
        }
        if (tid == 0) {
            sh.can_add = 1; sh.do_remove = 0; sh.k = -1; sh.l = -1; sh.choice = -1; sh.chosen_flat = -1;
            sh.found_flat = 0x7fffffffffffffffLL;
            const int ry = (MODE == LOOP_DIRECTED ? S.n : 0) + sh.y;
            sh.n_i = S.rlen[sh.x] + S.selfl[sh.x] + 1;                        // successors of x (:45 / :48) [+ x itself if it
            sh.n_j = S.rlen[ry] + S.selfl[ry] + 1;                            //  has a self-loop in G], then x (:46 / :49)
        }
        __syncthreads();
        const int x = sh.x, y = sh.y;
        const int n_i = sh.n_i, n_j = sh.n_j;
        const long long cells = (long long)n_i * n_j;
        if (cells > S.imp_cap || n_i > S.row_cap_max || n_j > S.row_cap_max) {
            if (tid == 0) sh.status = STATUS_TOO_MANY_CANDIDATES;
            __syncthreads();
            break;
        }
        SDRF_TICK(0);   // argmin/argmax
        // ---- 2. candidate matrix in networkx order (:45-54) and improvements (:57-62) ------------------
        const CandList nbI{S.ord, S.rstart[x], n_i, x};
        const CandList nbJ{S.ord, S.rstart[(MODE == LOOP_DIRECTED ? S.n : 0) + y], n_j, y};
        {
            const float cxy = sh.cxy;
            uint32_t* imp = S.imp;
            auto put = [=](int I, int J, float d) {    // (the classical flavour puts the improvement itself)
                imp[(long long)I * n_j + J] = (d == MASKED_D) ? IMP_MASKED
                                              : __float_as_uint(MODE == LOOP_CLASSICAL ? d : __fsub_rn(d, cxy));
            };
            double cxy_d = 0.0;
            if constexpr (PAPER) cxy_d = sh.cxy_d;
            score_pair<MODE>(S, g, gin, x, y, nbI, nbJ, sc, put, reinterpret_cast<unsigned long long*>(S.imp), cxy_d,
                             &sh, &dsh, dred, [&] { SDRF_TICK(7); });   // (profile build: scoring = prepare [7] + cells [1])
        }
        __syncthreads();
        SDRF_TICK(1);   // scoring
        // ---- 3. selection ------------------------------------------------------------------------------
        // thread t owns the contiguous flat range [t*L, (t+1)*L): counts and prefix sums follow candidate order
        const long long L = (cells + SDRF_THREADS - 1) / SDRF_THREADS;
        const long long f_lo = min(cells, (long long)tid * L), f_hi = min(cells, f_lo + L);
        // one pass: candidate count and (finite tau) the softmax weights exp(a*tau) of softmax.py:9
        const bool forced = (it == 0 && forced_choice >= 0);
        const bool weigh = !tau_inf;
        long long my_cnt = 0;
        double local = 0.0;
        int bad = 0;
        for (long long f = f_lo; f < f_hi; ++f) {
            const Bits bits = imp_at(f);
            if (bits == MASKED) continue;
            ++my_cnt;
            if (weigh) {
                const double e = exp(__dmul_rn((double)imp_val(bits), tau));
                if (!(e <= 1.7976931348623157e308)) bad = 1;   // inf or NaN
                local = __dadd_rn(local, e);
            }
        }
        long long n_cand, my_off;
        double total, carry;
        block_exscan_pair(my_cnt, local, &my_off, &carry, &n_cand, &total, &sh.red);
        const int nbad = __syncthreads_or(bad);
        if (tid == 0) sh.n_cand = n_cand;
        if (n_cand > 0) {
            if (draws >= n_uniforms) {
                if (tid == 0) sh.status = DCR_SDRF_NO_UNIFORM;
                __syncthreads();
                break;
            }
            const double u = uniforms[draws];
            if (forced) {
                if (forced_choice >= my_off && forced_choice < my_off + my_cnt) {
                    long long c = my_off;
                    for (long long f = f_lo; f < f_hi; ++f) {
                        if (imp_at(f) == MASKED) continue;
                        if (c == forced_choice) { sh.chosen_flat = f; sh.choice = (int)c; break; }
                        ++c;
                    }
                }
                __syncthreads();
                if (sh.chosen_flat < 0) {   // forced index out of range
                    if (tid == 0) sh.status = DCR_SDRF_NEED_HOST;
                    __syncthreads();
                    break;
                }
            } else if (tau_inf) {
                // softmax.py:5-8: one-hot at the first maximum; the draw then returns that index for any u in [0,1)
                BestT<Val> b{(Val)INFINITY, ~0ull};
                for (long long f = f_lo; f < f_hi; ++f) {
                    const Bits bits = imp_at(f);
                    if (bits == MASKED) continue;
                    b = best_of(b, BestT<Val>{-imp_val(bits), (unsigned long long)f});
                }
                b = block_best(b, &sh.red);
                const long long fstar = (long long)b.key;
                if (fstar >= f_lo && fstar < f_hi) {
                    long long c = my_off;
                    for (long long f = f_lo; f < fstar; ++f) c += imp_at(f) != MASKED;
                    sh.chosen_flat = fstar;
                    sh.choice = (int)c;
                }
                __syncthreads();
            } else {
                // softmax.py:9-10 + np.random.choice: p = exp(a*tau)/sum; first index whose normalised CDF > u
                if (nbad != 0 || total == 0.0 || !(total <= 1.7976931348623157e308)) {
                    // exp overflow -> inf/inf = NaN, all-underflow -> 0/0 = NaN (numpy: "probabilities contain
                    // NaN"); a finite-term sum that overflows gives p = 0 everywhere ("do not sum to 1")
                    if (tid == 0) sh.status = (nbad != 0 || total == 0.0) ? DCR_SDRF_PROB_NAN : DCR_SDRF_PROB_SUM;
                    __syncthreads();
                    break;
                }
                long long found = cells;   // first flat index in my range whose CDF exceeds u
                double below = 0.0, above = 0.0;
                long long c = my_off, found_c = 0;
                double run = carry;
                for (long long f = f_lo; f < f_hi; ++f) {
                    const Bits bits = imp_at(f);
                    if (bits == MASKED) continue;
                    const double e = exp(__dmul_rn((double)imp_val(bits), tau));
                    const double prev = run;
                    run = __dadd_rn(run, e);
                    if (__ddiv_rn(run, total) > u) {
                        found = f; found_c = c;
                        below = __ddiv_rn(prev, total);
                        above = __ddiv_rn(run, total);
                        break;
                    }
                    ++c;
                }
                if (found < cells) atomicMin(&sh.found_flat, found);
                __syncthreads();
                if (found < cells && sh.found_flat == found) {
                    sh.chosen_flat = found;
                    sh.choice = (int)found_c;
                    sh.below = below;
                    sh.above = above;
                }
                __syncthreads();
                // u within `guard` of a CDF boundary (or, by rounding, beyond the last one): numpy's exp / summation
                // order could decide differently -> hand the decision to the host with the improvements
                const bool near_boundary = sh.chosen_flat < 0 ||
                                           (guard > 0.0 && ((sh.above - u) < guard || (u - sh.below) < guard));
                if (near_boundary) {
                    long long cc = my_off;
                    for (long long f = f_lo; f < f_hi; ++f) {
                        const Bits bits = imp_at(f);
                        if (bits == MASKED) continue;
                        S.pend[cc++] = (double)imp_val(bits);
                    }
                    if (tid == 0) sh.status = DCR_SDRF_NEED_HOST;
                    __syncthreads();
                    break;
                }
            }
            ++draws;
            if (tid == 0) {
                const long long f = sh.chosen_flat;
                const int ck = nbI((int)(f / n_j)), cl = nbJ((int)(f % n_j));
                const bool swap = NX_LOOP && ck > cl;                            // sorted(...) (sdrf_no_cuda.py:37,50)
                sh.k = swap ? cl : ck;
                sh.l = swap ? ck : cl;
            }
        } else {
            if (tid == 0) { sh.can_add = 0; if (!remove_edges) sh.stop = 1; }   // :74-77
        }
        __syncthreads();
        SDRF_TICK(2);   // selection
        // ---- removal decision on the SAME C_t (:79-91) --------------------------------------------------
        if (tid == 0 && remove_edges && !sh.stop) {
            // BFC: fp32 compare, torch casts the Python float (:83); classical: Python int > float (sdrf_no_cuda.py:62);
            // paper: Python float > float
            bool above;
            if constexpr (PAPER) above = sh.cmax_d > bound64;
            else above = (MODE == LOOP_CLASSICAL) ? ((double)sh.cmax > bound64) : (sh.cmax > bound32);
            if (above) {
                if (sh.have_max) sh.do_remove = (MODE == LOOP_CLASSICAL && sh.xr == sh.yr) ? 3 : 1;   // 3: the maximum is a loop edge
                else if (!NX_LOOP && S.selfl[0]) sh.do_remove = 2;   // (0,0) fallback and G has the loop 0-0: it goes
                else sh.status = DCR_SDRF_REMOVE_NONEDGE;                // (0,0) fallback beat a negative bound
            } else if (!sh.can_add) {
                sh.stop = 1;
            }
        }
        __syncthreads();
        if (sh.status != DCR_SDRF_OK) break;
        // ---- 4. apply the edits, exact supports, dirty set ---------------------------------------------
        if (tid == 0) { dirty_count = 0; work_count = 0; }
        __syncthreads();
        const int k = sh.k, l = sh.l;
        if (k >= 0) {                                   // :69-73
            if (!edge_insert<MODE>(S, k, l)) {
                if (tid == 0) sh.status = DCR_SDRF_ARENA_FULL;
                __syncthreads();
                break;
            }
            SDRF_TICK(3);   // insert rows
            toggle_mark<MODE>(S, g, k, l, +1, &dirty_count, &sh);
            SDRF_TICK(4);   // supports + dirty (add)
        }
        if (sh.do_remove == 2) {                        // G.remove_edge(0, 0): only the insertion-order rows change (A[0,0] = 0 already)
            for (int row = 0; row <= (MODE == LOOP_DIRECTED ? S.n : 0); row += max(S.n, 1)) {   // node 0's row(s)
                ord_erase(S, S.rstart[row], S.rlen[row] + 1, 0, &sh);
                if (tid == 0) S.selfl[row] = 0;
                __syncthreads();
            }
        } else if (sh.do_remove == 3) {                 // classical loop: G.remove_edge(u, u) — degree - 2, u no longer its own neighbour
            const int u = sh.xr, start = S.rstart[u], len = S.rlen[u];
            ord_erase(S, start, len + 1, u, &sh);
            if (tid == 0) S.selfl[u] = 0;
            __syncthreads();
            for (int t = tid; t < len; t += SDRF_THREADS) {                 // every edge at u changes
                const int w = S.col[start + t];
                push_dirty(S, &dirty_count, min(u, w), max(u, w));
            }
            __syncthreads();
        } else if (sh.do_remove) {                      // :84-88
            const int xr = sh.xr, yr = sh.yr;
            toggle_mark<MODE>(S, g, xr, yr, -1, &dirty_count, &sh);
            edge_delete<MODE>(S, xr, yr, &sh);
        }
        SDRF_TICK(5);   // removal: supports + delete rows
        // ---- 5. refresh the curvature of the dirty edges ----------------------------------------------
        const int nd = min(dirty_count, S.dirty_cap);
        if (dirty_count > S.dirty_cap) {
            if (tid == 0) sh.status = DCR_SDRF_ARENA_FULL;
            __syncthreads();
            break;
        }
        refresh_dirty<MODE>(S, g, gin, nd, &work_count);
        SDRF_TICK(6);   // refresh
        // ---- 6. log ------------------------------------------------------------------------------------
        if (tid == 0) {
            int32_t* rec = log + (long long)it * DCR_SDRF_LOG_INTS;
            rec[0] = x; rec[1] = y; rec[2] = (int)n_cand; rec[3] = sh.k; rec[4] = sh.l; rec[5] = sh.choice;
            rec[6] = sh.do_remove ? sh.xr : -1;
            rec[7] = sh.do_remove ? sh.yr : -1;
        }
        __syncthreads();
        if (sh.stop) { ++it; break; }
    }
    __syncthreads();
    if (tid == 0) {
        result->status = sh.status;
        result->iterations_done = it;
        result->draws_used = draws;
        result->stopped = sh.stop;
        result->pending_n = sh.status == DCR_SDRF_NEED_HOST ? (int)sh.n_cand : 0;
        result->pending_x = sh.x;
        result->pending_y = sh.y;
        result->reserved = 0;
    }
}

template <int MODE>
__global__ void __launch_bounds__(SDRF_THREADS, 1)
sdrf_loop_kernel(SdrfDev S, int loops, int remove_edges, float bound32, double bound64, double tau, int tau_inf,
                 const double* __restrict__ uniforms, long long n_uniforms, int forced_choice, double guard,
                 int32_t* __restrict__ log, dcr_sdrf_result* __restrict__ result) {
    sdrf_loop_body<MODE, true>(S, loops, remove_edges, bound32, bound64, tau, tau_inf, uniforms, n_uniforms,
                               forced_choice, guard, log, result);
}

// Per-run arguments of the batch kernel (dcr_sdrf_run_batch packs one per run into the caller's workspace).
struct SdrfBatchDesc {
    SdrfDev S;
    int loops, forced_choice, tau_inf;
    float bound32;
    double bound64, tau;
    const double* uniforms;
    long long n_uniforms;
    int32_t* log;
    dcr_sdrf_result* result;
};
static_assert(sizeof(SdrfBatchDesc) % 8 == 0, "descriptor copied as 8-byte words");

// B independent runs, one CTA each (gridDim.x = B; CTAs beyond one per SM run in later waves).  The descriptor is
// copied to shared memory once, so the arena pointers are read from there rather than from global memory on every use.
template <int MODE>
__global__ void __launch_bounds__(SDRF_THREADS, 1)
sdrf_batch_loop_kernel(const SdrfBatchDesc* __restrict__ descs, int remove_edges, double guard) {
    __shared__ SdrfBatchDesc d;
    constexpr int WORDS = sizeof(SdrfBatchDesc) / 8;
    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(descs + blockIdx.x);
    if (threadIdx.x < WORDS) reinterpret_cast<unsigned long long*>(&d)[threadIdx.x] = src[threadIdx.x];
    __syncthreads();
    sdrf_loop_body<MODE, false>(d.S, d.loops, remove_edges, d.bound32, d.bound64, d.tau, d.tau_inf, d.uniforms,
                                d.n_uniforms, d.forced_choice, guard, d.log, d.result);
}

// Caller edits (dcr_sdrf_edit): edits[3t .. 3t+2] = (op, u, v), op 1 = G.add_edge(u, v), 0 = G.remove_edge(u, v),
// applied in order on one CTA.  Each edit is the loop's own toggle (edge_insert / edge_delete, toggle_mark) followed by
// the refresh of its dirty edges before the next edit: one toggle per refresh keeps the dirty list within dirty_cap.
// An add of a present edge changes nothing (networkx keeps its position).  The kernel stops BEFORE an edit with
// u == v or an id outside [0, n) (BAD_EDIT), a remove of an absent edge (REMOVE_NONEDGE) or an add beyond the
// additions budget (ARENA_FULL; scalars[2] counts the add edits, no-op adds included, scalars[3] is max_additions).
// Block-uniform arguments only: the single-state kernel and every CTA of the batch kernel run this on their own state.
template <int MODE>
__device__ __forceinline__ void sdrf_edit_body(const SdrfDev& S, const int32_t* __restrict__ edits, long long count,
                                               dcr_sdrf_result* __restrict__ result) {
    __shared__ LoopShared sh;
    __shared__ int dirty_count, work_count;
    const GraphView g{S.rstart, S.rlen, S.col};                 // undirected adjacency / successors
    const GraphView gin{S.rstart + S.n, S.rlen + S.n, S.col};   // predecessors (directed flavour only)
    int adds = S.scalars[2];                                    // block-uniform copies of the budget words
    const int add_limit = S.scalars[3];
    int status = DCR_SDRF_OK, u = -1, v = -1;
    long long t = 0;
    for (; t < count; ++t) {
        const int op = edits[3 * t];
        u = edits[3 * t + 1];
        v = edits[3 * t + 2];
        if ((op != 0 && op != 1) || u == v || u < 0 || u >= S.n || v < 0 || v >= S.n) { status = DCR_SDRF_BAD_EDIT; break; }
        const bool present = edge_slot(g, u, v) >= 0;
        if (op == 1 && adds >= add_limit) { status = DCR_SDRF_ARENA_FULL; break; }
        if (op == 0 && !present) { status = DCR_SDRF_REMOVE_NONEDGE; break; }
        adds += op;
        if (op == 1 && present) continue;
        if (threadIdx.x == 0) { dirty_count = 0; work_count = 0; }
        __syncthreads();
        if (op == 1) {
            if (!edge_insert<MODE>(S, u, v)) { status = DCR_SDRF_ARENA_FULL; break; }   // (not within the budget)
            toggle_mark<MODE>(S, g, u, v, +1, &dirty_count, &sh);
        } else {
            toggle_mark<MODE>(S, g, u, v, -1, &dirty_count, &sh);
            edge_delete<MODE>(S, u, v, &sh);
        }
        if (dirty_count > S.dirty_cap) { status = DCR_SDRF_ARENA_FULL; ++t; break; }   // (not within the budget)
        refresh_dirty<MODE>(S, g, gin, dirty_count, &work_count);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        S.scalars[2] = adds;
        result->status = status;
        result->iterations_done = (int)t;
        result->draws_used = 0;
        result->stopped = 0;
        result->pending_n = 0;
        result->pending_x = status == DCR_SDRF_OK ? -1 : u;
        result->pending_y = status == DCR_SDRF_OK ? -1 : v;
        result->reserved = 0;
    }
}

template <int MODE>
__global__ void __launch_bounds__(SDRF_THREADS, 1)
sdrf_edit_kernel(SdrfDev S, const int32_t* __restrict__ edits, long long count, dcr_sdrf_result* __restrict__ result) {
    sdrf_edit_body<MODE>(S, edits, count, result);
}

// Per-state arguments of the batched edit kernel (dcr_sdrf_edit_batch packs one per run into the caller's workspace).
struct SdrfEditDesc {
    SdrfDev S;
    const int32_t* edits;
    long long count;
    dcr_sdrf_result* result;
};
static_assert(sizeof(SdrfEditDesc) % 8 == 0, "descriptor copied as 8-byte words");

// B independent edit lists, one CTA per state, the descriptor copied to shared memory as in sdrf_batch_loop_kernel.
template <int MODE>
__global__ void __launch_bounds__(SDRF_THREADS, 1)
sdrf_batch_edit_kernel(const SdrfEditDesc* __restrict__ descs) {
    __shared__ SdrfEditDesc d;
    constexpr int WORDS = sizeof(SdrfEditDesc) / 8;
    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(descs + blockIdx.x);
    if (threadIdx.x < WORDS) reinterpret_cast<unsigned long long*>(&d)[threadIdx.x] = src[threadIdx.x];
    __syncthreads();
    sdrf_edit_body<MODE>(d.S, d.edits, d.count, d.result);
}

// ------------------------------------------------------------------------------------------------------------
// caller queries: the candidate scores of many pairs (dcr_sdrf_score_sizes, dcr_sdrf_score)
// ------------------------------------------------------------------------------------------------------------
// The pairs the loop itself can score: BFC and directed any 0 <= x, y < n (its (0,0) fallback scores a non-edge and
// x == y); classical an edge in either orientation or the loop edge (u, u) of a node that lists itself; paper an edge.
template <int MODE>
__device__ __forceinline__ bool score_query_ok(const SdrfDev& S, const GraphView& g, int x, int y) {
    if (x < 0 || x >= S.n || y < 0 || y >= S.n) return false;
    if constexpr (MODE == LOOP_BFC || MODE == LOOP_DIRECTED) return true;
    if (x == y) return MODE == LOOP_CLASSICAL && S.selfl[x];
    return edge_slot(g, x, y) >= 0;
}
// DCR_SDRF_OK and (n_i, n_j) of a query the score kernel takes, else its status
template <int MODE>
__device__ __forceinline__ int score_query_sizes(const SdrfDev& S, const GraphView& g, int x, int y, int& n_i, int& n_j) {
    n_i = n_j = 0;
    if (!score_query_ok<MODE>(S, g, x, y)) return DCR_SDRF_BAD_QUERY;
    const int a = cand_count(S, x), b = cand_count(S, (MODE == LOOP_DIRECTED ? S.n : 0) + y);
    if (a > S.row_cap_max || b > S.row_cap_max) return DCR_SDRF_TOO_MANY_CANDIDATES;   // (rows grown past the budget)
    n_i = a;
    n_j = b;
    return DCR_SDRF_OK;
}

template <int MODE>
__global__ void sdrf_score_sizes_kernel(SdrfDev S, const int32_t* __restrict__ pairs, int count,
                                        int32_t* __restrict__ sizes, int32_t* __restrict__ status) {
    const GraphView g{S.rstart, S.rlen, S.col};
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < count; q += gridDim.x * blockDim.x) {
        int n_i, n_j;
        status[q] = score_query_sizes<MODE>(S, g, pairs[2 * q], pairs[2 * q + 1], n_i, n_j);
        sizes[2 * q] = n_i;
        sizes[2 * q + 1] = n_j;
    }
}

// Persistent grid: CTA b scores the queries b, b + gridDim.x, ... with the loop's own scoring step (score_pair) on its
// slice of the caller's workspace (four scratch rows of `stride` ints).  Query q writes its candidate ids (nbI, then
// nbJ) at cand + cand_offsets[q], its n_i x n_j fp64 cells at imp + cell_offsets[q] (IMP_MASKED64 = masked) and one
// best record.  The state is only read: S arrives with its scratch pointers cleared (dcr_sdrf_score) and this copy's
// score scratch points into the workspace.
template <int MODE>
__global__ void __launch_bounds__(SDRF_THREADS, 1)
sdrf_score_kernel(SdrfDev S, const int32_t* __restrict__ pairs, int count, const int64_t* __restrict__ cell_offsets,
                  const int64_t* __restrict__ cand_offsets, int32_t* __restrict__ cand, unsigned long long* imp,
                  dcr_sdrf_score_best* __restrict__ best, int32_t* __restrict__ workspace, int stride) {
    constexpr bool PAPER = MODE == LOOP_PAPER;
    __shared__ std::conditional_t<PAPER, LoopSharedPaper, LoopShared> sh;
    __shared__ DirScoreShared dsh;
    __shared__ int dred[2];
    const int tid = threadIdx.x;
    const GraphView g{S.rstart, S.rlen, S.col};
    const GraphView gin{S.rstart + S.n, S.rlen + S.n, S.col};
    int32_t* ws = workspace + (long long)blockIdx.x * 4 * stride;   // this CTA's scratch: the copy S points at it
    S.base1 = ws;
    S.base2 = ws + stride;
    S.posI = ws + 2 * stride;
    S.posJ = ws + 3 * stride;
    const ScoreScratch sc{S.base1, S.base2, S.posI, S.posJ};
    for (int q = blockIdx.x; q < count; q += gridDim.x) {
        const int x = pairs[2 * q], y = pairs[2 * q + 1];
        dcr_sdrf_score_best* rec = best + q;
        int n_i, n_j;
        if (score_query_sizes<MODE>(S, g, x, y, n_i, n_j) != DCR_SDRF_OK) {   // (the sizes pass reported it)
            if (tid == 0) *rec = {-1, -1, -1, -1, __longlong_as_double(-1ll)};
            continue;
        }
        const CandList nbI{S.ord, S.rstart[x], n_i, x};
        const CandList nbJ{S.ord, S.rstart[(MODE == LOOP_DIRECTED ? S.n : 0) + y], n_j, y};
        int32_t* cq = cand + cand_offsets[q];
        for (int t = tid; t < n_i + n_j; t += SDRF_THREADS) cq[t] = t < n_i ? nbI(t) : nbJ(t - n_i);
        // C[x,y] of the state; 0 for a non-edge (the loop's (0,0) fallback, the reference's dense C)
        const int sxy = edge_slot(g, x, y);
        const float cxy = (!PAPER && sxy >= 0) ? S.c32[sxy] : 0.0f;
        double cxy_d = 0.0;
        if constexpr (PAPER) cxy_d = paper_get(S, sxy);               // (a paper query is an edge)
        unsigned long long* out = imp + cell_offsets[q];
        auto put = [=](int I, int J, float d) {    // the value the loop draws from, as fp64
            out[(long long)I * n_j + J] =
                d == MASKED_D ? IMP_MASKED64
                              : (unsigned long long)__double_as_longlong(MODE == LOOP_CLASSICAL ? d : __fsub_rn(d, cxy));
        };
        score_pair<MODE>(S, g, gin, x, y, nbI, nbJ, sc, put, out, cxy_d, &sh, &dsh, dred, [] {});
        __syncthreads();
        // the best record: the first maximum in cell order (the loop's tau = inf selection) and its rank among the
        // unmasked cells; thread t owns the contiguous cell range [t*L, (t+1)*L) as in the loop
        const long long cells = (long long)n_i * n_j;
        const long long L = (cells + SDRF_THREADS - 1) / SDRF_THREADS;
        const long long f_lo = min(cells, (long long)tid * L), f_hi = min(cells, f_lo + L);
        long long my_cnt = 0;
        BestT<double> b{(double)INFINITY, ~0ull};
        for (long long f = f_lo; f < f_hi; ++f) {
            const unsigned long long bits = out[f];
            if (bits == IMP_MASKED64) continue;
            ++my_cnt;
            b = best_of(b, BestT<double>{-__longlong_as_double((long long)bits), (unsigned long long)f});
        }
        long long n_cand;
        const long long my_off = block_exscan_ll(my_cnt, &n_cand, &sh.red);
        b = block_best(b, &sh.red);
        const long long fstar = (long long)b.key;
        if (n_cand == 0) {
            if (tid == 0) *rec = {0, -1, -1, -1, __longlong_as_double(-1ll)};
        } else if (fstar >= f_lo && fstar < f_hi) {
            long long c = my_off;
            for (long long f = f_lo; f < fstar; ++f) c += out[f] != IMP_MASKED64;
            *rec = {n_cand, c, nbI((int)(fstar / n_j)), nbJ((int)(fstar % n_j)), __longlong_as_double((long long)out[fstar])};
        }
        __syncthreads();
    }
}

// the kernels of the loop flavour that runs DCR_SDRF_MODE_* `mode`
struct LoopKernels {
    decltype(&sdrf_init_curvature_kernel<LOOP_BFC>) init;
    decltype(&sdrf_loop_kernel<LOOP_BFC>) single;
    decltype(&sdrf_batch_loop_kernel<LOOP_BFC>) batch;
    decltype(&sdrf_edit_kernel<LOOP_BFC>) edit;
    decltype(&sdrf_batch_edit_kernel<LOOP_BFC>) batch_edit;
    decltype(&sdrf_score_sizes_kernel<LOOP_BFC>) score_sizes;
    decltype(&sdrf_score_kernel<LOOP_BFC>) score;
    decltype(&sdrf_batch_init_curvature_kernel<LOOP_BFC>) batch_init;
};
template <int MODE>
static LoopKernels loop_kernels_of() {
    return {sdrf_init_curvature_kernel<MODE>, sdrf_loop_kernel<MODE>, sdrf_batch_loop_kernel<MODE>,
            sdrf_edit_kernel<MODE>, sdrf_batch_edit_kernel<MODE>, sdrf_score_sizes_kernel<MODE>,
            sdrf_score_kernel<MODE>, sdrf_batch_init_curvature_kernel<MODE>};
}
static LoopKernels loop_kernels(int mode) {
    switch (mode) {
    case DCR_SDRF_MODE_BFC: return loop_kernels_of<LOOP_BFC>();
    case DCR_SDRF_MODE_BFC_DIRECTED: return loop_kernels_of<LOOP_DIRECTED>();
    case DCR_SDRF_MODE_BFC_PAPER: return loop_kernels_of<LOOP_PAPER>();
    default: return loop_kernels_of<LOOP_CLASSICAL>();
    }
}

// ------------------------------------------------------------------------------------------------------------
// export
// ------------------------------------------------------------------------------------------------------------
// with_self: row lengths of the INSERTION-ORDER rows (a node that lists itself has one entry more)
__device__ __forceinline__ int export_row_len(const SdrfDev& S, int v, int with_self) {
    return S.rlen[v] + (with_self ? S.selfl[v] : 0);
}
__global__ void sdrf_export_rowptr_kernel(SdrfDev S, int32_t* rowptr, int with_self) {
    __shared__ Reduce red;
    // single CTA: chunked exclusive scan of rlen
    const int n = S.n;
    const int L = (n + SDRF_THREADS - 1) / SDRF_THREADS;
    const int lo = min(n, (int)threadIdx.x * L), hi = min(n, lo + L);
    long long s = 0;
    for (int v = lo; v < hi; ++v) s += export_row_len(S, v, with_self);
    long long total;
    long long off = block_exscan_ll(s, &total, &red);
    for (int v = lo; v < hi; ++v) { rowptr[v] = (int32_t)off; off += export_row_len(S, v, with_self); }
    if (threadIdx.x == 0) rowptr[n] = (int32_t)total;
}
__global__ void sdrf_export_order_kernel(SdrfDev S, const int32_t* rowptr, int32_t* order_out) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int v = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < S.n; v += warps) {
        const int s = S.rstart[v], d = S.rlen[v] + S.selfl[v], o = rowptr[v];
        for (int t = lane; t < d; t += 32) order_out[o + t] = S.ord[s + t];
    }
}
__global__ void sdrf_export_rows_kernel(SdrfDev S, const int32_t* rowptr, int32_t* order_out, int32_t* colidx,
                                        float* c32, int32_t* tri) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int v = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < S.n; v += warps) {
        const int s = S.rstart[v], d = S.rlen[v], o = rowptr[v];
        for (int t = lane; t < d; t += 32) {
            if (order_out) order_out[o + t] = S.ord[s + t];
            if (colidx) colidx[o + t] = S.col[s + t];
            if (c32) c32[o + t] = S.c32[s + t];
            if (tri) tri[o + t] = S.supp[s + t];
        }
    }
}
__global__ void sdrf_export_c64_kernel(SdrfDev S, const int32_t* rowptr, double* c64) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int v = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < S.n; v += warps) {
        const int s = S.rstart[v], d = S.rlen[v], o = rowptr[v];
        for (int t = lane; t < d; t += 32) c64[o + t] = paper_get(S, s + t);
    }
}
// from_networkx(G).edge_index of the insertion-order rows (G.from_networkx_order): row w lists its neighbours < w
// ascending, which is the prefix of its sorted arena row, then its neighbours >= w (its self entry included) in insertion
// order.  directed: the successor rows as they are (G.from_digraph_order).  One warp per row; `rowptr` comes from
// sdrf_export_rowptr_kernel(with_self = 1).  Nothing is written at or beyond `capacity`.
// Row w of one state, written from column o on with the node ids shifted by `shift` (the batched export's node offset).
__device__ __forceinline__ void export_edge_row(const SdrfDev& S, int w, long long o, long long shift, int64_t* src,
                                                int64_t* dst, long long capacity, int directed, int lane) {
    const int s = S.rstart[w], len = S.rlen[w], olen = len + S.selfl[w];
    const int lo = directed ? 0 : lower_bound(S.col, s, len, w);
    for (int t = lane; t < lo; t += 32)
        if (o + t < capacity) { src[o + t] = w + shift; dst[o + t] = S.col[s + t] + shift; }
    o += lo;
    for (int base = 0; base < olen; base += 32) {
        const int t = base + lane;
        const int x = t < olen ? S.ord[s + t] : -1;
        const bool keep = t < olen && (directed || x >= w);
        const unsigned m = __ballot_sync(FULL, keep);
        const long long p = o + __popc(m & ((1u << lane) - 1u));
        if (keep && p < capacity) { src[p] = w + shift; dst[p] = x + shift; }
        o += __popc(m);
    }
}
__global__ void sdrf_export_edge_index_kernel(SdrfDev S, const int32_t* rowptr, int64_t* src, int64_t* dst,
                                              long long capacity, int directed) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < S.n; w += warps)
        export_edge_row(S, w, rowptr[w], 0, src, dst, capacity, directed, lane);
}

// ---- the batched export (dcr_sdrf_export_edge_index_batch): all states' rows in three launches
struct SdrfExportDesc {
    SdrfDev S;
    long long node_offset;    // added to every node id of the state
};
static_assert(sizeof(SdrfExportDesc) % 8 == 0, "descriptor table packed as 8-byte words");

// 1. counts[r] = export_row_len of global row r (row_off[b] = sum over earlier states of n)
__global__ void sdrf_batch_export_counts_kernel(const SdrfExportDesc* __restrict__ descs,
                                                const long long* __restrict__ row_off, int count,
                                                long long* __restrict__ counts) {
    for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < row_off[count];
         r += (long long)gridDim.x * blockDim.x) {
        const int b = state_of(row_off, count, r);
        counts[r] = export_row_len(descs[b].S, (int)(r - row_off[b]), 1);
    }
}
// 2. single CTA: counts[0 .. R) becomes its exclusive prefix (in place), edge_ptr[b] = the first column of state b and
//    edge_ptr[count] = the total
__global__ void __launch_bounds__(SDRF_THREADS, 1)
sdrf_batch_export_scan_kernel(const long long* __restrict__ row_off, int count, long long* counts,
                              int64_t* __restrict__ edge_ptr) {
    __shared__ Reduce red;
    const long long R = row_off[count];
    const long long L = (R + SDRF_THREADS - 1) / SDRF_THREADS;
    const long long lo = min(R, (long long)threadIdx.x * L), hi = min(R, lo + L);
    long long s = 0;
    for (long long r = lo; r < hi; ++r) s += counts[r];
    long long total;
    long long off = block_exscan_ll(s, &total, &red);
    for (long long r = lo; r < hi; ++r) { const long long c = counts[r]; counts[r] = off; off += c; }
    __syncthreads();
    for (int b = threadIdx.x; b < count; b += SDRF_THREADS) edge_ptr[b] = row_off[b] < R ? counts[row_off[b]] : total;
    if (threadIdx.x == 0) edge_ptr[count] = total;
}
// 3. one warp per global row, from column rowptr[r]
__global__ void sdrf_batch_export_rows_kernel(const SdrfExportDesc* __restrict__ descs,
                                              const long long* __restrict__ row_off, int count,
                                              const long long* __restrict__ rowptr, int64_t* src, int64_t* dst,
                                              long long capacity, int directed) {
    const int lane = threadIdx.x & 31;
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; r < row_off[count]; r += warps) {
        const int b = state_of(row_off, count, r);
        const SdrfExportDesc& d = descs[b];
        export_edge_row(d.S, (int)(r - row_off[b]), rowptr[r], d.node_offset, src, dst, capacity, directed, lane);
    }
}
__global__ void sdrf_copy_pending_kernel(const double* pend, double* out, long long n) {
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x)
        out[t] = pend[t];
}

}  // namespace dcr

using namespace dcr;

// Slabs of the states of one dcr_sdrf_create_batch call live in one allocation; each state holds a reference and the
// last dcr_sdrf_destroy frees it.
struct SdrfPool {
    void* base;
    std::atomic<int> refs;
};

struct dcr_sdrf {
    SdrfDev dev;
    void* slab;           // one allocation backing every array (a pooled state: its part of the pool)
    size_t slab_bytes;
    int mode;             // DCR_SDRF_MODE_*
    int64_t n_self;       // nodes that list themselves (self-loops of G)
    SdrfPool* pool;       // null: the state owns `slab`
};

template <class T>
static T* carve(char*& p, size_t count) {
    T* out = (T*)p;
    p += (count * sizeof(T) + 255) / 256 * 256;
    return out;
}

// Points D's arrays into the slab at `p` (D's sizes set).  The persistent state, rstart … scalars, is carved first and
// the scratch after it, so the state is the byte prefix [slab, D.base1) of the slab: that prefix is all dcr_sdrf_fork
// copies.  A new array that must survive between launches goes before base1.
static void carve_slab(SdrfDev& D, char* p, int rows, bool paper) {
    D.rstart = carve<int32_t>(p, rows); D.rlen = carve<int32_t>(p, rows); D.rcap = carve<int32_t>(p, rows);
    D.selfl = carve<int32_t>(p, rows);
    D.col = carve<int32_t>(p, D.cap_total); D.ord = carve<int32_t>(p, D.cap_total);
    D.supp = carve<int32_t>(p, D.cap_total); D.c32 = carve<float>(p, D.cap_total);
    D.owner = carve<int32_t>(p, D.cap_total); D.flag = carve<int32_t>(p, D.cap_total);
    D.scalars = carve<int32_t>(p, 8);
    // ---- scratch of one launch (not copied by dcr_sdrf_fork)
    D.base1 = carve<int32_t>(p, D.row_cap_max); D.base2 = carve<int32_t>(p, D.row_cap_max);
    D.posI = carve<int32_t>(p, D.row_cap_max); D.posJ = carve<int32_t>(p, D.row_cap_max);
    D.imp = carve<uint32_t>(p, (paper ? 2 : 1) * D.imp_cap); D.pend = carve<double>(p, D.imp_cap);
    D.dirty = carve<int32_t>(p, (size_t)2 * D.dirty_cap); D.work = carve<int32_t>(p, D.dirty_cap);
    D.wlist = carve<int32_t>(p, D.row_cap_max);
}
static size_t persistent_bytes(const dcr_sdrf* s) { return (size_t)((char*)s->dev.base1 - (char*)s->slab); }

// The host image and the sizes of one state, from its insertion-order rows: the validation and sizing shared by
// dcr_sdrf_create_mode and dcr_sdrf_create_batch.
struct SdrfPlan {
    SdrfDev D;            // the sizes (n, ctype, cap_total, row_cap_max, imp_cap, dirty_cap); no pointers yet
    int rows;
    int64_t sum_cap;      // arena slots filled at set-up
    int64_t n_self;
    size_t bytes;         // slab size
    std::vector<int32_t> rstart, rlen, rcap, selfl, col, ord, owner;
    int32_t scal[8];
};

// rows [0,n): the neighbour (directed: successor) lists, rows [n,2n): the predecessor lists (directed mode only);
// row_len(r) / row_src(r) give row r, nnz / in_nnz the entries of the two halves.  `who` starts every error message.
template <class RowLen, class RowSrc>
static int sdrf_plan(const char* who, int n, int mode, int64_t nnz, int64_t in_nnz, RowLen row_len, RowSrc row_src,
                     int64_t max_additions, SdrfPlan& P) {
    const bool directed = mode == DCR_SDRF_MODE_BFC_DIRECTED;
    const bool paper = mode == DCR_SDRF_MODE_BFC_PAPER;
    const int rows = directed ? 2 * n : n;
    if (directed && in_nnz != nnz) { set_error("%s: successor / predecessor lists disagree", who); return 1; }
    std::vector<int32_t> rstart(rows), rlen(rows), rcap(rows), selfl(rows, 0);
    int64_t sum_cap = 0, n_self = 0;
    int d1 = 0, d2 = 0;   // the two largest row lengths
    for (int v = 0; v < rows; ++v) {
        int len = row_len(v);
        {                                              // a node may list ITSELF once (a self-loop of G; A has none):
            const int32_t* src = row_src(v);           // insertion-order row only (directed: successor AND predecessor row)
            const int me = v < n ? v : v - n;
            int hits = 0;
            for (int t = 0; t < len; ++t) hits += src[t] == me;
            if (hits > 1) { set_error("%s: node %d lists itself more than once", who, me); return 1; }
            if (hits && paper) { set_error("%s: node %d lists itself (the paper-flavour loop takes no self-loops)", who, me); return 1; }
            selfl[v] = hits;
            if (v < n) n_self += hits;                 // (counted once per node: the successor / neighbour rows)
            len -= hits;
        }
        const int cap = len + selfl[v] + std::max(2, len / 8);
        rstart[v] = (int32_t)sum_cap;
        rlen[v] = len;
        rcap[v] = cap;
        sum_cap += cap;
        if (len > d1) { d2 = d1; d1 = len; } else if (len > d2) d2 = len;
    }
    const int64_t cap_total = 5 * sum_cap + 8 * max_additions + 1024;
    if (cap_total > 0x7ffffff0LL) { set_error("%s: graph too large for a 32-bit arena", who); return 1; }
    std::vector<int32_t> col(sum_cap, 0), ord(sum_cap, 0), owner(sum_cap, -1);
    nnz -= n_self;                            // (directed: successor entries; the predecessor rows mirror them)
    for (int v = 0; v < rows; ++v) {
        const int len = rlen[v];
        const int32_t* src = row_src(v);
        const int self = v < n ? v : v - n;
        int filled = 0;
        for (int t = 0; t < len + selfl[v]; ++t) {
            if (src[t] < 0 || src[t] >= n || (src[t] == self && !selfl[v])) { set_error("%s: bad neighbour id", who); return 1; }
            ord[rstart[v] + t] = src[t];
            if (src[t] == self) continue;
            col[rstart[v] + filled] = src[t];
            owner[rstart[v] + filled] = v;
            ++filled;
        }
        std::sort(col.begin() + rstart[v], col.begin() + rstart[v] + len);
        for (int t = 1; t < len; ++t)
            if (col[rstart[v] + t] == col[rstart[v] + t - 1]) { set_error("%s: duplicate neighbour", who); return 1; }
    }
    if (directed) {   // the predecessor rows must be the transpose of the successor rows
        for (int v = 0; v < n; ++v)
            if (selfl[v] != selfl[n + v]) { set_error("%s: successor / predecessor lists disagree", who); return 1; }
        for (int v = 0; v < n; ++v)
            for (int t = 0; t < rlen[v]; ++t) {
                const int w = col[rstart[v] + t];
                const int32_t* b = col.data() + rstart[n + w];
                if (!std::binary_search(b, b + rlen[n + w], v)) {
                    set_error("%s: successor / predecessor lists disagree", who);
                    return 1;
                }
            }
    }
    SdrfDev& D = P.D;
    D = SdrfDev{};
    D.n = n;
    D.ctype = (mode >= DCR_SDRF_MODE_1D && mode <= DCR_SDRF_MODE_HAANTJES) ? mode - DCR_SDRF_MODE_1D : 0;
    D.cap_total = (int)cap_total;
    const int64_t row_cap_max = (int64_t)d1 + max_additions + 2;
    D.row_cap_max = (int)std::min<int64_t>(row_cap_max, 0x7ffffff0LL);
    // candidate matrix: (deg x + 1)(deg y + 1) <= the product of the two longest rows after all additions
    D.imp_cap = std::min<int64_t>(((int64_t)d1 + max_additions + 2) * ((int64_t)d2 + max_additions + 2), (int64_t)1 << 28);
    // dirty pairs of one iteration: two toggles, each at most the entries at four rows + the closing edges (paper loop:
    // the entries at k and l + at most one pair per directed entry, so 2 nnz per toggle, paper_mark_dirty)
    D.dirty_cap = (int)std::min<int64_t>(4 * (nnz + 2 * max_additions) + 4096, 0x3ffffff0LL);
    size_t bytes = 0;
    auto add = [&](size_t count, size_t elem) { bytes += (count * elem + 255) / 256 * 256; };
    add(rows, 4); add(rows, 4); add(rows, 4); add(rows, 4);  // rstart rlen rcap selfl
    for (int i = 0; i < 6; ++i) add(cap_total, 4);           // col ord supp c32 owner flag
    add(8, 4);                                               // scalars
    for (int i = 0; i < 4; ++i) add(D.row_cap_max, 4);       // base1 base2 posI posJ
    add(D.imp_cap, paper ? 8 : 4); add(D.imp_cap, 8);        // imp, pend
    add((size_t)2 * D.dirty_cap, 4); add(D.dirty_cap, 4);    // dirty, work
    add(D.row_cap_max, 4);                                   // wlist
    P.rows = rows;
    P.sum_cap = sum_cap;
    P.n_self = n_self;
    P.bytes = bytes;
    P.rstart = std::move(rstart); P.rlen = std::move(rlen); P.rcap = std::move(rcap); P.selfl = std::move(selfl);
    P.col = std::move(col); P.ord = std::move(ord); P.owner = std::move(owner);
    // [0] arena top, [1] nnz, [2] add edits so far, [3] their limit (dcr_sdrf_edit)
    const int32_t scal[8] = {(int32_t)sum_cap, (int32_t)nnz, 0, (int32_t)std::min<int64_t>(max_additions, 0x7fffffff), 0, 0, 0, 0};
    std::copy(scal, scal + 8, P.scal);
    return 0;
}

static int sdrf_create_impl(int n, int mode, const int32_t* rowptr_host, const int32_t* order_host,
                            const int32_t* in_rowptr_host, const int32_t* in_order_host, int64_t max_additions,
                            dcr_sdrf** out) {
    if (n <= 0 || !rowptr_host || !out) { set_error("dcr_sdrf_create: bad arguments"); return 1; }
    if (mode < DCR_SDRF_MODE_BFC || mode > DCR_SDRF_MODE_BFC_PAPER) { set_error("dcr_sdrf_create: unknown mode"); return 1; }
    const bool directed = mode == DCR_SDRF_MODE_BFC_DIRECTED;
    const bool paper = mode == DCR_SDRF_MODE_BFC_PAPER;
    if (directed && !in_rowptr_host) { set_error("dcr_sdrf_create: the directed mode needs the predecessor lists"); return 1; }
    auto row_len = [&](int r) { return r < n ? rowptr_host[r + 1] - rowptr_host[r] : in_rowptr_host[r - n + 1] - in_rowptr_host[r - n]; };
    auto row_src = [&](int r) { return r < n ? order_host + rowptr_host[r] : in_order_host + in_rowptr_host[r - n]; };
    SdrfPlan P;
    if (sdrf_plan("dcr_sdrf_create", n, mode, rowptr_host[n], directed ? in_rowptr_host[n] : 0, row_len, row_src,
                  max_additions, P))
        return 1;
    const int rows = P.rows;
    const int64_t sum_cap = P.sum_cap, cap_total = P.D.cap_total;
    dcr_sdrf* s = new dcr_sdrf();
    s->mode = mode;
    s->n_self = P.n_self;
    s->pool = nullptr;
    SdrfDev& D = s->dev;
    D = P.D;
    cudaError_t e = cudaMalloc(&s->slab, P.bytes);
    if (e != cudaSuccess) { delete s; return cuda_fail(e, "cudaMalloc(sdrf slab)", __FILE__, __LINE__); }
    s->slab_bytes = P.bytes;
    carve_slab(D, (char*)s->slab, rows, paper);

    auto fail = [&](cudaError_t err, const char* what) {
        cudaFree(s->slab);
        delete s;
        return cuda_fail(err, what, __FILE__, __LINE__);
    };
#define SDRF_TRY(call) do { cudaError_t e2 = (call); if (e2 != cudaSuccess) return fail(e2, #call); } while (0)
    SDRF_TRY(cudaMemcpy(D.rstart, P.rstart.data(), rows * 4, cudaMemcpyHostToDevice));
    SDRF_TRY(cudaMemcpy(D.rlen, P.rlen.data(), rows * 4, cudaMemcpyHostToDevice));
    SDRF_TRY(cudaMemcpy(D.rcap, P.rcap.data(), rows * 4, cudaMemcpyHostToDevice));
    SDRF_TRY(cudaMemcpy(D.selfl, P.selfl.data(), rows * 4, cudaMemcpyHostToDevice));
    SDRF_TRY(cudaMemset(D.owner, 0xff, cap_total * 4));
    SDRF_TRY(cudaMemset(D.flag, 0, cap_total * 4));
    SDRF_TRY(cudaMemset(D.supp, 0, cap_total * 4));
    SDRF_TRY(cudaMemset(D.c32, 0, cap_total * 4));
    if (sum_cap > 0) {
        SDRF_TRY(cudaMemcpy(D.col, P.col.data(), sum_cap * 4, cudaMemcpyHostToDevice));
        SDRF_TRY(cudaMemcpy(D.ord, P.ord.data(), sum_cap * 4, cudaMemcpyHostToDevice));
        SDRF_TRY(cudaMemcpy(D.owner, P.owner.data(), sum_cap * 4, cudaMemcpyHostToDevice));
    }
    SDRF_TRY(cudaMemcpy(D.scalars, P.scal, sizeof(P.scal), cudaMemcpyHostToDevice));
    if (sum_cap > 0) {
        const int ctas = (int)std::min<int64_t>((sum_cap + 7) / 8, (int64_t)sm_count() * 8);
        if (!directed && !paper) sdrf_init_support_kernel<<<ctas, 256>>>(D, (int)sum_cap);   // (paper: no supports)
        loop_kernels(mode).init<<<ctas, 256>>>(D, (int)sum_cap);
        SDRF_TRY(cudaGetLastError());
    }
    SDRF_TRY(cudaDeviceSynchronize());
#undef SDRF_TRY
    *out = s;
    return 0;
}

// Every state's slab is carved out of one pool allocation at a 256-byte aligned offset.  The host images of all states go
// to the device in one copy of a packed staging buffer (a stream-ordered allocation freed after the set-up), whose tail
// holds the device tables; three launches then fill the slabs, the supports and the curvature of every state.
extern "C" int dcr_sdrf_create_batch(int count, int mode, const int32_t* num_nodes, const int64_t* rowptr_host,
                                     const int32_t* order_host, const int64_t* in_rowptr_host,
                                     const int32_t* in_order_host, const int64_t* max_additions, dcr_sdrf** out_host) {
    if (count < 1 || !num_nodes || !rowptr_host || !max_additions || !out_host) {
        set_error("dcr_sdrf_create_batch: bad arguments (count must be >= 1)");
        return 1;
    }
    if (mode < DCR_SDRF_MODE_BFC || mode > DCR_SDRF_MODE_BFC_PAPER) { set_error("dcr_sdrf_create_batch: unknown mode"); return 1; }
    const bool directed = mode == DCR_SDRF_MODE_BFC_DIRECTED;
    const bool paper = mode == DCR_SDRF_MODE_BFC_PAPER;
    if (directed && !in_rowptr_host) { set_error("dcr_sdrf_create_batch: the directed mode needs the predecessor lists"); return 1; }
    // node offsets; the row offsets must start at 0 and never decrease
    std::vector<int64_t> node_off(count + 1, 0);
    for (int g = 0; g < count; ++g) {
        if (num_nodes[g] <= 0) { set_error("dcr_sdrf_create_batch: graph %d has %d nodes", g, num_nodes[g]); return 1; }
        if (max_additions[g] < 0) { set_error("dcr_sdrf_create_batch: graph %d: max_additions < 0", g); return 1; }
        node_off[g + 1] = node_off[g] + num_nodes[g];
    }
    const int64_t N = node_off[count];
    for (int half = 0; half < (directed ? 2 : 1); ++half) {
        const int64_t* rp = half ? in_rowptr_host : rowptr_host;
        if (rp[0] != 0) { set_error("dcr_sdrf_create_batch: row offsets must start at 0"); return 1; }
        for (int64_t v = 0; v < N; ++v)
            if (rp[v + 1] < rp[v] || rp[v + 1] - rp[v] > 0x7fffffff) {
                const int64_t g = std::upper_bound(node_off.begin(), node_off.end(), v) - node_off.begin() - 1;
                set_error("dcr_sdrf_create_batch: graph %lld: the row offsets decrease at node %lld", (long long)g,
                          (long long)(v - node_off[g]));
                return 1;
            }
    }
    if ((rowptr_host[N] > 0 && !order_host) || (directed && in_rowptr_host[N] > 0 && !in_order_host)) {
        set_error("dcr_sdrf_create_batch: bad arguments (no neighbour lists)");
        return 1;
    }
    std::vector<SdrfPlan> plans(count);
    for (int g = 0; g < count; ++g) {
        const int n = num_nodes[g];
        const int64_t* rp = rowptr_host + node_off[g];
        const int64_t* irp = directed ? in_rowptr_host + node_off[g] : nullptr;
        auto row_len = [&](int r) { return (int)(r < n ? rp[r + 1] - rp[r] : irp[r - n + 1] - irp[r - n]); };
        auto row_src = [&](int r) { return r < n ? order_host + rp[r] : in_order_host + irp[r - n]; };
        char who[64];
        snprintf(who, sizeof(who), "dcr_sdrf_create_batch: graph %d", g);
        if (sdrf_plan(who, n, mode, rp[n] - rp[0], directed ? irp[n] - irp[0] : 0, row_len, row_src, max_additions[g],
                      plans[g]))
            return 1;
    }
    // pool offsets (every slab size is a multiple of 256), staging offsets (int32 words) and the device tables
    std::vector<size_t> slab_off(count + 1, 0);
    std::vector<int64_t> stage_off(count + 1, 0);
    std::vector<long long> unit_off(count + 1, 0), entry_off(count + 1, 0);
    for (int g = 0; g < count; ++g) {
        const SdrfPlan& P = plans[g];
        slab_off[g + 1] = slab_off[g] + P.bytes;
        stage_off[g + 1] = stage_off[g] + 4 * (int64_t)P.rows + 3 * P.sum_cap + 8;
        unit_off[g + 1] = unit_off[g] + P.D.cap_total + P.rows;
        entry_off[g + 1] = entry_off[g] + P.sum_cap;
    }
    const size_t words = (size_t)(stage_off[count] + 1) / 2 * 2;                 // (8-byte aligned tables after it)
    const size_t table_bytes = sizeof(SdrfInitDesc) * count + 2 * sizeof(long long) * (count + 1);
    const size_t stage_bytes = 4 * words + table_bytes;
    void* pool_base = nullptr;
    cudaError_t e = cudaMalloc(&pool_base, slab_off[count]);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(sdrf pool)", __FILE__, __LINE__);
    std::vector<char> host(stage_bytes);
    int32_t* hw = reinterpret_cast<int32_t*>(host.data());
    SdrfInitDesc* hdesc = reinterpret_cast<SdrfInitDesc*>(host.data() + 4 * words);
    long long* hunit = reinterpret_cast<long long*>(hdesc + count);
    long long* hentry = hunit + count + 1;
    void* stage = nullptr;
    e = cudaMallocAsync(&stage, stage_bytes, 0);
    if (e != cudaSuccess) { cudaFree(pool_base); return cuda_fail(e, "cudaMallocAsync(sdrf staging)", __FILE__, __LINE__); }
    const int32_t* dstage = reinterpret_cast<const int32_t*>(stage);
    for (int g = 0; g < count; ++g) {
        const SdrfPlan& P = plans[g];
        int32_t* w = hw + stage_off[g];
        for (const std::vector<int32_t>* a : {&P.rstart, &P.rlen, &P.rcap, &P.selfl, &P.col, &P.ord, &P.owner}) {
            std::copy(a->begin(), a->end(), w);
            w += a->size();
        }
        std::copy(P.scal, P.scal + 8, w);
        SdrfInitDesc& d = hdesc[g];
        d.S = P.D;
        carve_slab(d.S, (char*)pool_base + slab_off[g], P.rows, paper);
        d.stage = dstage + stage_off[g];
        d.rows = P.rows;
        d.used = (int)P.sum_cap;
    }
    std::copy(unit_off.begin(), unit_off.end(), hunit);
    std::copy(entry_off.begin(), entry_off.end(), hentry);
    const SdrfInitDesc* ddesc = reinterpret_cast<const SdrfInitDesc*>((char*)stage + 4 * words);
    const long long* dunit = reinterpret_cast<const long long*>(ddesc + count);
    const long long* dentry = dunit + count + 1;
    e = cudaMemcpyAsync(stage, host.data(), stage_bytes, cudaMemcpyHostToDevice, 0);
    if (e == cudaSuccess) {
        const int ctas = (int)std::max<int64_t>(1, std::min<int64_t>((unit_off[count] + 255) / 256, (int64_t)sm_count() * 8));
        sdrf_batch_setup_kernel<<<ctas, 256>>>(ddesc, dunit, count);
        if (entry_off[count] > 0) {
            const int ictas = (int)std::min<int64_t>((entry_off[count] + 7) / 8, (int64_t)sm_count() * 8);
            if (!directed && !paper) sdrf_batch_init_support_kernel<<<ictas, 256>>>(ddesc, dentry, count);
            loop_kernels(mode).batch_init<<<ictas, 256>>>(ddesc, dentry, count);
        }
        e = cudaGetLastError();
    }
    const cudaError_t ef = cudaFreeAsync(stage, 0);
    if (e == cudaSuccess) e = ef;
    const cudaError_t es = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = es;
    if (e != cudaSuccess) { cudaFree(pool_base); return cuda_fail(e, "dcr_sdrf_create_batch: set-up", __FILE__, __LINE__); }
    SdrfPool* pool = new SdrfPool{pool_base, {count}};
    for (int g = 0; g < count; ++g) {
        dcr_sdrf* s = new dcr_sdrf();
        s->dev = hdesc[g].S;
        s->slab = (char*)pool_base + slab_off[g];
        s->slab_bytes = plans[g].bytes;
        s->mode = mode;
        s->n_self = plans[g].n_self;
        s->pool = pool;
        out_host[g] = s;
    }
    return 0;
}

extern "C" int dcr_sdrf_create(int n, const int32_t* rowptr_host, const int32_t* order_host, int64_t max_additions,
                               dcr_sdrf** out) {
    return sdrf_create_impl(n, DCR_SDRF_MODE_BFC, rowptr_host, order_host, nullptr, nullptr, max_additions, out);
}

extern "C" int dcr_sdrf_create_mode(int n, int mode, const int32_t* rowptr_host, const int32_t* order_host,
                                    const int32_t* in_rowptr_host, const int32_t* in_order_host,
                                    int64_t max_additions, dcr_sdrf** out) {
    return sdrf_create_impl(n, mode, rowptr_host, order_host, in_rowptr_host, in_order_host, max_additions, out);
}

extern "C" void dcr_sdrf_destroy(dcr_sdrf* s) {
    if (!s) return;
    if (!s->pool) cudaFree(s->slab);
    else if (s->pool->refs.fetch_sub(1) == 1) {
        cudaFree(s->pool->base);
        delete s->pool;
    }
    delete s;
}

// Every copy gets a slab of the source's size (same sizes, so the same carve) and one device-to-device copy of the
// persistent prefix on `stream`; the scratch is not copied.  All slabs are allocated before any copy is enqueued, so a
// failure leaves nothing behind.
extern "C" int dcr_sdrf_fork(dcr_sdrf* s, int count, dcr_sdrf** out_host, void* stream) {
    if (!s || count < 1 || !out_host) { set_error("dcr_sdrf_fork: bad arguments"); return 1; }
    const bool directed = s->mode == DCR_SDRF_MODE_BFC_DIRECTED;
    const bool paper = s->mode == DCR_SDRF_MODE_BFC_PAPER;
    std::vector<dcr_sdrf*> copies;
    auto release = [&]() {
        for (dcr_sdrf* c : copies) { cudaFree(c->slab); delete c; }
    };
    for (int b = 0; b < count; ++b) {
        dcr_sdrf* c = new dcr_sdrf(*s);
        c->pool = nullptr;                      // (a copy owns its slab, also when the source is pooled)
        const cudaError_t e = cudaMalloc(&c->slab, s->slab_bytes);
        if (e != cudaSuccess) { delete c; release(); return cuda_fail(e, "cudaMalloc(sdrf fork slab)", __FILE__, __LINE__); }
        copies.push_back(c);
        carve_slab(c->dev, (char*)c->slab, directed ? 2 * s->dev.n : s->dev.n, paper);
    }
    const size_t bytes = persistent_bytes(s);
    for (dcr_sdrf* c : copies) {
        const cudaError_t e = cudaMemcpyAsync(c->slab, s->slab, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
        if (e != cudaSuccess) { release(); return cuda_fail(e, "cudaMemcpyAsync(sdrf fork)", __FILE__, __LINE__); }
    }
    for (int b = 0; b < count; ++b) out_host[b] = copies[b];
    return 0;
}

extern "C" int dcr_sdrf_run(dcr_sdrf* s, int loops, int remove_edges, double removal_bound, double tau,
                            const double* uniforms, int64_t n_uniforms, int forced_choice, double guard, int32_t* log,
                            dcr_sdrf_result* result, void* stream) {
    if (!s || !result || (loops > 0 && !log)) { set_error("dcr_sdrf_run: bad arguments"); return 1; }
    const int tau_inf = std::isinf(tau) && tau > 0;
    loop_kernels(s->mode).single<<<1, SDRF_THREADS, 0, (cudaStream_t)stream>>>(
        s->dev, loops, remove_edges, (float)removal_bound, removal_bound, tau, tau_inf, uniforms, (long long)n_uniforms,
        forced_choice, guard, log, result);
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int dcr_sdrf_edit(dcr_sdrf* s, const int32_t* edits, int64_t count, dcr_sdrf_result* result, void* stream) {
    if (!s || !result || count < 0 || (count > 0 && !edits)) { set_error("dcr_sdrf_edit: bad arguments"); return 1; }
    loop_kernels(s->mode).edit<<<1, SDRF_THREADS, 0, (cudaStream_t)stream>>>(s->dev, edits, (long long)count, result);
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t dcr_sdrf_edit_batch_workspace_bytes(int count) {
    return count < 1 ? 0 : (int64_t)count * (int64_t)sizeof(SdrfEditDesc);
}

extern "C" int dcr_sdrf_edit_batch(const dcr_sdrf_edit_run* runs, int count, void* workspace, int64_t workspace_bytes,
                                   void* stream) {
    if (count < 1 || !runs) { set_error("dcr_sdrf_edit_batch: count must be >= 1"); return 1; }
    std::vector<SdrfEditDesc> descs(count);
    std::vector<const dcr_sdrf*> seen(count);
    for (int b = 0; b < count; ++b) {
        const dcr_sdrf_edit_run& r = runs[b];
        if (!r.state) { set_error("dcr_sdrf_edit_batch: run %d has no state", b); return 1; }
        if (!r.result || r.count < 0 || (r.count > 0 && !r.edits)) {
            set_error("dcr_sdrf_edit_batch: run %d: bad arguments", b);
            return 1;
        }
        if (r.state->mode != runs[0].state->mode) {
            set_error("dcr_sdrf_edit_batch: run %d has loop mode %d, run 0 has %d (one mode per call)", b, r.state->mode,
                      runs[0].state->mode);
            return 1;
        }
        descs[b] = {r.state->dev, r.edits, (long long)r.count, r.result};
        seen[b] = r.state;
    }
    std::sort(seen.begin(), seen.end());
    if (std::adjacent_find(seen.begin(), seen.end()) != seen.end()) {
        set_error("dcr_sdrf_edit_batch: the same state appears twice (runs of one call must own their states)");
        return 1;
    }
    if (!workspace || workspace_bytes < dcr_sdrf_edit_batch_workspace_bytes(count)) {
        set_error("dcr_sdrf_edit_batch: workspace of dcr_sdrf_edit_batch_workspace_bytes(%d) = %lld bytes required", count,
                  (long long)dcr_sdrf_edit_batch_workspace_bytes(count));
        return 1;
    }
    if ((uintptr_t)workspace % alignof(SdrfEditDesc)) { set_error("dcr_sdrf_edit_batch: workspace must be 8-byte aligned"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    // pageable source: the copy is staged before cudaMemcpyAsync returns, so `descs` may go out of scope
    DCR_CUDA(cudaMemcpyAsync(workspace, descs.data(), sizeof(SdrfEditDesc) * count, cudaMemcpyHostToDevice, st));
    loop_kernels(runs[0].state->mode).batch_edit<<<count, SDRF_THREADS, 0, st>>>((const SdrfEditDesc*)workspace);
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t dcr_sdrf_batch_workspace_bytes(int count) {
    return count < 1 ? 0 : (int64_t)count * (int64_t)sizeof(SdrfBatchDesc);
}

extern "C" int dcr_sdrf_run_batch(const dcr_sdrf_batch_run* runs, int count, int remove_edges, double guard,
                                  void* workspace, int64_t workspace_bytes, void* stream) {
    if (count < 1 || !runs) { set_error("dcr_sdrf_run_batch: count must be >= 1"); return 1; }
    std::vector<SdrfBatchDesc> descs(count);
    std::vector<const dcr_sdrf*> seen(count);
    for (int b = 0; b < count; ++b) {
        const dcr_sdrf_batch_run& r = runs[b];
        if (!r.state) { set_error("dcr_sdrf_run_batch: run %d has no state", b); return 1; }
        if (!r.result || (r.loops > 0 && !r.log)) { set_error("dcr_sdrf_run_batch: run %d: bad arguments", b); return 1; }
        if (r.state->mode != runs[0].state->mode) {
            set_error("dcr_sdrf_run_batch: run %d has loop mode %d, run 0 has %d (one mode per call)", b, r.state->mode,
                      runs[0].state->mode);
            return 1;
        }
        SdrfBatchDesc& d = descs[b];
        d.S = r.state->dev;
        d.loops = r.loops;
        d.forced_choice = r.forced_choice;
        d.tau_inf = std::isinf(r.tau) && r.tau > 0;
        d.bound32 = (float)r.removal_bound;
        d.bound64 = r.removal_bound;
        d.tau = r.tau;
        d.uniforms = r.uniforms;
        d.n_uniforms = (long long)r.n_uniforms;
        d.log = r.log;
        d.result = r.result;
        seen[b] = r.state;
    }
    std::sort(seen.begin(), seen.end());
    if (std::adjacent_find(seen.begin(), seen.end()) != seen.end()) {
        set_error("dcr_sdrf_run_batch: the same state appears twice (runs of one call must own their states)");
        return 1;
    }
    if (!workspace || workspace_bytes < dcr_sdrf_batch_workspace_bytes(count)) {
        set_error("dcr_sdrf_run_batch: workspace of dcr_sdrf_batch_workspace_bytes(%d) = %lld bytes required", count,
                  (long long)dcr_sdrf_batch_workspace_bytes(count));
        return 1;
    }
    if ((uintptr_t)workspace % alignof(SdrfBatchDesc)) { set_error("dcr_sdrf_run_batch: workspace must be 8-byte aligned"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    // pageable source: the copy is staged before cudaMemcpyAsync returns, so `descs` may go out of scope
    DCR_CUDA(cudaMemcpyAsync(workspace, descs.data(), sizeof(SdrfBatchDesc) * count, cudaMemcpyHostToDevice, st));
    loop_kernels(runs[0].state->mode).batch<<<count, SDRF_THREADS, 0, st>>>((const SdrfBatchDesc*)workspace,
                                                                             remove_edges, guard);
    DCR_LAUNCH_CHECK();
    return 0;
}

// ints per scratch row of one CTA of sdrf_score_kernel (every candidate list is at most row_cap_max long)
static int score_stride(const dcr_sdrf* s) { return (s->dev.row_cap_max + 63) / 64 * 64; }

extern "C" int64_t dcr_sdrf_score_workspace_bytes(dcr_sdrf* s, int count) {
    if (!s || count < 1) return 0;
    return (int64_t)std::min(count, sm_count()) * 4 * score_stride(s) * (int64_t)sizeof(int32_t);
}

extern "C" int dcr_sdrf_score_sizes(dcr_sdrf* s, const int32_t* pairs, int count, int32_t* sizes, int32_t* status,
                                    void* stream) {
    if (!s || count < 1 || !pairs || !sizes || !status) { set_error("dcr_sdrf_score_sizes: bad arguments"); return 1; }
    const int ctas = std::max(1, std::min((count + 255) / 256, sm_count() * 8));
    loop_kernels(s->mode).score_sizes<<<ctas, 256, 0, (cudaStream_t)stream>>>(s->dev, pairs, count, sizes, status);
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int dcr_sdrf_score(dcr_sdrf* s, const int32_t* pairs, int count, const int64_t* cell_offsets,
                              const int64_t* cand_offsets, int32_t* cand, double* imp, dcr_sdrf_score_best* best,
                              void* workspace, int64_t workspace_bytes, void* stream) {
    if (!s || count < 1 || !pairs || !cell_offsets || !cand_offsets || !cand || !imp || !best) {
        set_error("dcr_sdrf_score: bad arguments");
        return 1;
    }
    if (!workspace || workspace_bytes < dcr_sdrf_score_workspace_bytes(s, count)) {
        set_error("dcr_sdrf_score: workspace of dcr_sdrf_score_workspace_bytes(state, %d) = %lld bytes required", count,
                  (long long)dcr_sdrf_score_workspace_bytes(s, count));
        return 1;
    }
    if ((uintptr_t)workspace % 4) { set_error("dcr_sdrf_score: workspace must be 4-byte aligned"); return 1; }
    // the kernel reads the state only: its copy has no scratch, so a write to the state's own scratch cannot happen
    SdrfDev D = s->dev;
    D.base1 = D.base2 = D.posI = D.posJ = D.dirty = D.work = D.wlist = nullptr;
    D.imp = nullptr;
    D.pend = nullptr;
    loop_kernels(s->mode).score<<<std::min(count, sm_count()), SDRF_THREADS, 0, (cudaStream_t)stream>>>(
        D, pairs, count, cell_offsets, cand_offsets, cand, reinterpret_cast<unsigned long long*>(imp), best,
        (int32_t*)workspace, score_stride(s));
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int dcr_sdrf_pending_improvements(dcr_sdrf* s, double* out, int64_t capacity, void* stream) {
    if (!s || !out) { set_error("dcr_sdrf_pending_improvements: bad arguments"); return 1; }
    if (capacity <= 0) return 0;
    const int64_t n = std::min<int64_t>(capacity, s->dev.imp_cap);
    sdrf_copy_pending_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 1024), 256, 0, (cudaStream_t)stream>>>(
        s->dev.pend, out, n);
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t dcr_sdrf_nnz(dcr_sdrf* s) {
    if (!s) return -1;
    int32_t scal[2] = {0, 0};
    if (cudaMemcpy(scal, s->dev.scalars, sizeof(scal), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return scal[1];
}

extern "C" int dcr_sdrf_export(dcr_sdrf* s, int32_t* rowptr, int32_t* order_out, int32_t* colidx_sorted,
                               float* c32_sorted, int32_t* tri_sorted, void* stream) {
    if (!s || !rowptr) { set_error("dcr_sdrf_export: bad arguments"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    if (order_out && s->n_self > 0) {
        set_error("dcr_sdrf_export: this state has nodes that list themselves; use dcr_sdrf_export_order for the "
                  "insertion-order rows");
        return 1;
    }
    sdrf_export_rowptr_kernel<<<1, SDRF_THREADS, 0, st>>>(s->dev, rowptr, 0);
    DCR_LAUNCH_CHECK();
    const int ctas = std::max(1, std::min((s->dev.n + 7) / 8, sm_count() * 8));
    sdrf_export_rows_kernel<<<ctas, 256, 0, st>>>(s->dev, rowptr, order_out, colidx_sorted, c32_sorted, tri_sorted);
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int dcr_sdrf_export_order(dcr_sdrf* s, int32_t* rowptr_order, int32_t* order_out, void* stream) {
    if (!s || !rowptr_order || !order_out) { set_error("dcr_sdrf_export_order: bad arguments"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    sdrf_export_rowptr_kernel<<<1, SDRF_THREADS, 0, st>>>(s->dev, rowptr_order, 1);
    DCR_LAUNCH_CHECK();
    const int ctas = std::max(1, std::min((s->dev.n + 7) / 8, sm_count() * 8));
    sdrf_export_order_kernel<<<ctas, 256, 0, st>>>(s->dev, rowptr_order, order_out);
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int dcr_sdrf_export_edge_index(dcr_sdrf* s, int32_t* rowptr_order, int64_t* src, int64_t* dst,
                                          int64_t capacity, void* stream) {
    if (!s || !rowptr_order || capacity < 0 || (capacity > 0 && (!src || !dst))) {
        set_error("dcr_sdrf_export_edge_index: bad arguments");
        return 1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    sdrf_export_rowptr_kernel<<<1, SDRF_THREADS, 0, st>>>(s->dev, rowptr_order, 1);
    DCR_LAUNCH_CHECK();
    const int ctas = std::max(1, std::min((s->dev.n + 7) / 8, sm_count() * 8));
    sdrf_export_edge_index_kernel<<<ctas, 256, 0, st>>>(s->dev, rowptr_order, src, dst, (long long)capacity,
                                                        s->mode == DCR_SDRF_MODE_BFC_DIRECTED);
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int64_t dcr_sdrf_export_edge_index_batch_workspace_bytes(dcr_sdrf* const* states, int count) {
    if (count < 1 || !states) return 0;
    int64_t rows = 0;
    for (int b = 0; b < count; ++b) {
        if (!states[b]) return 0;
        rows += states[b]->dev.n;
    }
    return (int64_t)sizeof(SdrfExportDesc) * count + (int64_t)sizeof(long long) * (count + 1 + rows);
}

extern "C" int dcr_sdrf_export_edge_index_batch(dcr_sdrf* const* states, int count, const int64_t* node_offsets,
                                                int64_t* src, int64_t* dst, int64_t capacity, int64_t* edge_ptr,
                                                void* workspace, int64_t workspace_bytes, void* stream) {
    if (count < 1 || !states || !node_offsets || !edge_ptr || capacity < 0 || (capacity > 0 && (!src || !dst))) {
        set_error("dcr_sdrf_export_edge_index_batch: bad arguments (count must be >= 1)");
        return 1;
    }
    // host tables: one descriptor per state, then the row offsets (count + 1); the device copy is followed by the
    // per-row counts, which the scan turns into the global column offsets
    std::vector<char> host(sizeof(SdrfExportDesc) * count + sizeof(long long) * (count + 1));
    SdrfExportDesc* desc = reinterpret_cast<SdrfExportDesc*>(host.data());
    long long* row_off = reinterpret_cast<long long*>(desc + count);
    row_off[0] = 0;
    for (int b = 0; b < count; ++b) {
        if (!states[b]) { set_error("dcr_sdrf_export_edge_index_batch: state %d is null", b); return 1; }
        if (states[b]->mode != states[0]->mode) {
            set_error("dcr_sdrf_export_edge_index_batch: state %d has loop mode %d, state 0 has %d (one mode per call)", b,
                      states[b]->mode, states[0]->mode);
            return 1;
        }
        if (node_offsets[b] < 0 || (b > 0 && node_offsets[b] < node_offsets[b - 1] + states[b - 1]->dev.n)) {
            set_error("dcr_sdrf_export_edge_index_batch: node_offsets[%d] = %lld overlaps the nodes of the state before "
                      "it or is negative", b, (long long)node_offsets[b]);
            return 1;
        }
        desc[b] = {states[b]->dev, (long long)node_offsets[b]};
        row_off[b + 1] = row_off[b] + states[b]->dev.n;
    }
    if (!workspace || workspace_bytes < dcr_sdrf_export_edge_index_batch_workspace_bytes(states, count)) {
        set_error("dcr_sdrf_export_edge_index_batch: workspace of dcr_sdrf_export_edge_index_batch_workspace_bytes = %lld "
                  "bytes required", (long long)dcr_sdrf_export_edge_index_batch_workspace_bytes(states, count));
        return 1;
    }
    if ((uintptr_t)workspace % 8) { set_error("dcr_sdrf_export_edge_index_batch: workspace must be 8-byte aligned"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    const SdrfExportDesc* ddesc = (const SdrfExportDesc*)workspace;
    const long long* drow_off = (const long long*)(ddesc + count);
    long long* rowptr = (long long*)(drow_off + count + 1);
    const long long rows = row_off[count];
    // pageable source: the copy is staged before cudaMemcpyAsync returns, so `host` may go out of scope
    DCR_CUDA(cudaMemcpyAsync(workspace, host.data(), host.size(), cudaMemcpyHostToDevice, st));
    const int ctas = (int)std::max<long long>(1, std::min<long long>((rows + 255) / 256, (long long)sm_count() * 8));
    sdrf_batch_export_counts_kernel<<<ctas, 256, 0, st>>>(ddesc, drow_off, count, rowptr);
    DCR_LAUNCH_CHECK();
    sdrf_batch_export_scan_kernel<<<1, SDRF_THREADS, 0, st>>>(drow_off, count, rowptr, edge_ptr);
    DCR_LAUNCH_CHECK();
    const int wctas = (int)std::max<long long>(1, std::min<long long>((rows + 7) / 8, (long long)sm_count() * 8));
    sdrf_batch_export_rows_kernel<<<wctas, 256, 0, st>>>(ddesc, drow_off, count, rowptr, src, dst, (long long)capacity,
                                                         states[0]->mode == DCR_SDRF_MODE_BFC_DIRECTED);
    DCR_LAUNCH_CHECK();
    return 0;
}

extern "C" int dcr_sdrf_export_c64(dcr_sdrf* s, int32_t* rowptr, double* c64_sorted, void* stream) {
    if (!s || !rowptr || !c64_sorted) { set_error("dcr_sdrf_export_c64: bad arguments"); return 1; }
    if (s->mode != DCR_SDRF_MODE_BFC_PAPER) { set_error("dcr_sdrf_export_c64: only DCR_SDRF_MODE_BFC_PAPER keeps fp64 values"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    sdrf_export_rowptr_kernel<<<1, SDRF_THREADS, 0, st>>>(s->dev, rowptr, 0);
    DCR_LAUNCH_CHECK();
    const int ctas = std::max(1, std::min((s->dev.n + 7) / 8, sm_count() * 8));
    sdrf_export_c64_kernel<<<ctas, 256, 0, st>>>(s->dev, rowptr, c64_sorted);
    DCR_LAUNCH_CHECK();
    return 0;
}

#ifdef DCR_SDRF_PROFILE
extern "C" int dcr_sdrf_phase_cycles(unsigned long long* out_host, int reset) {
    if (cudaMemcpyFromSymbol(out_host, dcr::g_sdrf_phase, sizeof(unsigned long long) * 16) != cudaSuccess) return 1;
    if (reset) {
        unsigned long long zero[16] = {0};
        if (cudaMemcpyToSymbol(dcr::g_sdrf_phase, zero, sizeof(zero)) != cudaSuccess) return 1;
    }
    return 0;
}
#endif
