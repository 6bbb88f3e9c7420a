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
#include <cmath>
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
enum { LOOP_BFC = 0, LOOP_DIRECTED = 1, LOOP_CLASSICAL = 2 };

#ifndef DCR_SDRF_THREADS
#define DCR_SDRF_THREADS 1024
#endif
constexpr int SDRF_THREADS = DCR_SDRF_THREADS;
constexpr int SDRF_WARPS = SDRF_THREADS / 32;
constexpr uint32_t IMP_MASKED = 0xffffffffu;   // bit pattern marking a masked cell in the improvement matrix
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
    int32_t* owner;       // arena: row id of the slot, -1 = free
    int32_t* flag;        // arena: dedupe flags for the refresh
    int32_t* scalars;     // [0] arena_top, [1] nnz
    int32_t* base1; int32_t* base2; int32_t* posI; int32_t* posJ;   // score scratch [row_cap_max]
    uint32_t* imp;        // improvement matrix (fp32 bits)
    double* pend;         // compact improvements of a pending iteration
    int32_t* dirty;       // pairs (a,b): 2*dirty_cap ints
    int32_t* work;        // slots to refresh: dirty_cap ints
    int32_t* wlist;       // common-neighbour list scratch [row_cap_max]
};

// ------------------------------------------------------------------------------------------------------------
// block-wide primitives (SDRF_THREADS threads, every thread calls)
// ------------------------------------------------------------------------------------------------------------
struct Best { float v; unsigned long long key; };   // "smaller v wins, then smaller key"

__device__ __forceinline__ Best best_of(Best a, Best b) {
    return (b.v < a.v || (b.v == a.v && b.key < a.key)) ? b : a;
}
__device__ __forceinline__ Best warp_best(Best a) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        Best b;
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
    Best best;
};

__device__ Best block_best(Best a, Reduce* r) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    a = warp_best(a);
    if (lane == 0) { r->v[warp] = a.v; r->k[warp] = a.key; }
    __syncthreads();
    if (warp == 0) {
        Best b;
        b.v = lane < SDRF_WARPS ? r->v[lane] : INFINITY;
        b.key = lane < SDRF_WARPS ? r->k[lane] : ~0ull;
        b = warp_best(b);
        if (lane == 0) r->best = b;
    }
    __syncthreads();
    Best out = r->best;
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
// initialisation kernels over arena slots (multi-CTA)
// ------------------------------------------------------------------------------------------------------------
__global__ void sdrf_init_support_kernel(SdrfDev S, int top) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    GraphView g{S.rstart, S.rlen, S.col};
    for (int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; s < top; s += warps) {
        const int a = S.owner[s];
        if (a < 0) continue;
        const int c = warp_intersect_count(g, a, S.col[s], lane);
        if (lane == 0) S.supp[s] = c;
    }
}
template <int MODE>
__global__ void sdrf_init_curvature_kernel(SdrfDev S, int top) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; s < top; s += warps) {
        const int a = S.owner[s];
        if (a < 0) continue;
        float c;
        if constexpr (MODE == LOOP_DIRECTED) {
            if (a >= S.n) continue;                 // predecessor rows carry no curvature
            const GraphView gout{S.rstart, S.rlen, S.col}, gin{S.rstart + S.n, S.rlen + S.n, S.col};
            c = directed_entry_curvature(gout, gin, a, S.col[s], lane).c32;
        } else if constexpr (MODE == LOOP_CLASSICAL) {
            c = classical_curvature(S, a, S.col[s], s);
        } else {
            c = entry_curvature(S, a, S.col[s], s, lane);
        }
        if (lane == 0) S.c32[s] = c;
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
    __shared__ LoopShared sh;
    __shared__ DirScoreShared dsh;
    __shared__ int dirty_count, work_count, dred[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
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
        if constexpr (MODE == LOOP_CLASSICAL) {
            // ---- 1c. min(G.edges, key=curvature) / max(...) (sdrf_no_cuda.py:27, :59-61) --------------------
            // G.edges lists every edge once, from its first endpoint in node order, neighbours in insertion order:
            // the first minimum is at the smallest u that has an entry (u, v > u) with the minimal value, and among
            // those at the earliest position of u's insertion-order row.  The maximum is taken over the same C_t
            // (curv_dict predates the addition; the new edge is excluded, :59).
            float vmin = INFINITY, vmax = -INFINITY;
            for (int s = tid; s < top; s += SDRF_THREADS) {
                if (S.owner[s] < 0) continue;
                const float v = S.c32[s];
                vmin = fminf(vmin, v);
                vmax = fmaxf(vmax, v);
            }
            for (int u = tid; u < S.n; u += SDRF_THREADS) {     // the loop edges (u,u) of G.edges
                if (!S.selfl[u]) continue;
                const float v = classical_loop_curvature(S, u);
                vmin = fminf(vmin, v);
                vmax = fmaxf(vmax, v);
            }
            vmin = block_best(Best{vmin, 0ull}, &sh.red).v;
            vmax = -block_best(Best{-vmax, 0ull}, &sh.red).v;
            if (!(vmin <= vmax)) {                              // no edges: min() of an empty sequence
                if (tid == 0) sh.status = DCR_SDRF_EMPTY_GRAPH;
                __syncthreads();
                break;
            }
            unsigned long long umin = ~0ull, umax = ~0ull;
            for (int s = tid; s < top; s += SDRF_THREADS) {
                const int o = S.owner[s];
                if (o < 0 || S.col[s] < o) continue;
                const float v = S.c32[s];
                if (v == vmin) umin = min(umin, (unsigned long long)o);
                if (v == vmax) umax = min(umax, (unsigned long long)o);
            }
            for (int u = tid; u < S.n; u += SDRF_THREADS) {
                if (!S.selfl[u]) continue;
                const float v = classical_loop_curvature(S, u);
                if (v == vmin) umin = min(umin, (unsigned long long)u);
                if (v == vmax) umax = min(umax, (unsigned long long)u);
            }
            const int xu = (int)block_best(Best{0.0f, umin}, &sh.red).key;
            const int xru = (int)block_best(Best{0.0f, umax}, &sh.red).key;
            // this thread's first position in u's insertion-order row of an entry (u, v >= u) of value `val` (the row
            // holds the node itself where its loop was added: G.edges reports it there)
            auto first_pos = [&](int u, float val) {
                const int st = S.rstart[u], len = S.rlen[u];
                unsigned long long p = ~0ull;
                for (int t = tid; t < len + S.selfl[u]; t += SDRF_THREADS) {
                    const int v = S.ord[st + t];
                    const bool hit = v == u ? classical_loop_curvature(S, u) == val
                                            : (v > u && S.c32[find_sorted(S.col, st, len, v)] == val);
                    if (hit) p = min(p, (unsigned long long)t);
                }
                return p;
            };
            unsigned long long pmin = first_pos(xu, vmin), pmax = first_pos(xru, vmax);
            pmin = block_best(Best{0.0f, pmin}, &sh.red).key;
            pmax = block_best(Best{0.0f, pmax}, &sh.red).key;
            if (tid == 0) {
                sh.have_min = 1; sh.have_max = 1;
                sh.x = xu;  sh.y = S.ord[S.rstart[xu] + (int)pmin];   sh.cxy = vmin;
                sh.xr = xru; sh.yr = S.ord[S.rstart[xru] + (int)pmax]; sh.cmax = vmax;
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
        const int ox = S.rstart[x], oy = S.rstart[(MODE == LOOP_DIRECTED ? S.n : 0) + y];
        auto nbI = [=](int I) { return I < n_i - 1 ? S.ord[ox + I] : x; };
        auto nbJ = [=](int J) { return J < n_j - 1 ? S.ord[oy + J] : y; };
        {
            const float cxy = sh.cxy;
            uint32_t* imp = S.imp;
            auto put = [=](int I, int J, float d) {
                imp[(long long)I * n_j + J] = (d == MASKED_D) ? IMP_MASKED : __float_as_uint(__fsub_rn(d, cxy));
            };
            if constexpr (MODE == LOOP_BFC) {
                score_prepare(g, S.supp, x, y, nbI, n_i, nbJ, n_j, sc, &sh.score);
                SDRF_TICK(7);   // (profile build: scoring = prepare [7] + cells [1])
                // x (y) sits at the end of its list — and, with a self-loop, once more inside it: then every row is checked
                score_cells(g, S.supp, x, y, nbI, n_i, nbJ, n_j, sc, &sh.score, put, S.selfl[x] ? -1 : n_i - 1,
                            S.selfl[y] ? -1 : n_j - 1);
            } else if constexpr (MODE == LOOP_DIRECTED) {
                directed_score_prepare(g, gin, x, y, nbI, n_i, nbJ, n_j, sc, &dsh, dred);
                directed_score_cells(g, gin, x, y, nbI, n_i, nbJ, n_j, sc, &dsh, put);
            } else {
                // sdrf_no_cuda.py:41-46 in closed form: adding (i,j) changes curvature(x,y) only when it touches x or y.
                // i == x (then j in N(y)\N(x)): deg x + 1 and one more triangle; j == y mirrored; every other
                // candidate leaves both degrees and the common neighbours alone.
                const float special = S.ctype == 0 ? -1.0f : (S.ctype == 1 ? 2.0f : 1.0f);
                for (long long c = tid; c < cells; c += SDRF_THREADS) {
                    const int I = (int)(c / n_j), J = (int)(c - (long long)I * n_j);
                    const int i = nbI(I), j = nbJ(J);
                    const bool masked = (i == j) || edge_slot(g, i, j) >= 0;       // :34
                    imp[c] = masked ? IMP_MASKED : __float_as_uint((i == x || j == y) ? special : 0.0f);
                }
            }
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
            const uint32_t bits = S.imp[f];
            if (bits == IMP_MASKED) continue;
            ++my_cnt;
            if (weigh) {
                const double e = exp(__dmul_rn((double)__uint_as_float(bits), tau));
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
                        if (S.imp[f] == IMP_MASKED) continue;
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
                Best b{INFINITY, ~0ull};
                for (long long f = f_lo; f < f_hi; ++f) {
                    const uint32_t bits = S.imp[f];
                    if (bits == IMP_MASKED) continue;
                    b = best_of(b, Best{-__uint_as_float(bits), (unsigned long long)f});
                }
                b = block_best(b, &sh.red);
                const long long fstar = (long long)b.key;
                if (fstar >= f_lo && fstar < f_hi) {
                    long long c = my_off;
                    for (long long f = f_lo; f < fstar; ++f) c += S.imp[f] != IMP_MASKED;
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
                    const uint32_t bits = S.imp[f];
                    if (bits == IMP_MASKED) continue;
                    const double e = exp(__dmul_rn((double)__uint_as_float(bits), tau));
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
                        const uint32_t bits = S.imp[f];
                        if (bits == IMP_MASKED) continue;
                        S.pend[cc++] = (double)__uint_as_float(bits);
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
                const bool swap = (MODE == LOOP_CLASSICAL) && ck > cl;           // sorted(...) (sdrf_no_cuda.py:37,50)
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
            // BFC: fp32 compare, torch casts the Python float (:83); classical: Python int > float (sdrf_no_cuda.py:62)
            const bool above = (MODE == LOOP_CLASSICAL) ? ((double)sh.cmax > bound64) : (sh.cmax > bound32);
            if (above) {
                if (sh.have_max) sh.do_remove = (MODE == LOOP_CLASSICAL && sh.xr == sh.yr) ? 3 : 1;   // 3: the maximum is a loop edge
                else if (MODE != LOOP_CLASSICAL && S.selfl[0]) sh.do_remove = 2;   // (0,0) fallback and G has the loop 0-0: it goes
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
        constexpr int L_ROW = (MODE == LOOP_DIRECTED);  // directed: the mirror entry lives in the predecessor rows
        if (k >= 0) {                                   // :69-73
            bool ok = row_insert(S, k, l);
            ok = ok && row_insert(S, L_ROW * S.n + l, k);
            if (!ok) {
                if (tid == 0) sh.status = DCR_SDRF_ARENA_FULL;
                __syncthreads();
                break;
            }
            if (tid == 0) S.scalars[1] += L_ROW ? 1 : 2;
            __syncthreads();
            SDRF_TICK(3);   // insert rows
            if constexpr (MODE == LOOP_DIRECTED) directed_mark_dirty(S, k, l, &dirty_count);
            else toggle_supports<MODE == LOOP_BFC>(S, g, k, l, +1, &dirty_count, &sh);
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
            if constexpr (MODE == LOOP_DIRECTED) directed_mark_dirty(S, xr, yr, &dirty_count);
            else toggle_supports<MODE == LOOP_BFC>(S, g, xr, yr, -1, &dirty_count, &sh);
            row_delete(S, xr, yr, &sh);
            row_delete(S, L_ROW * S.n + yr, xr, &sh);
            if (tid == 0) S.scalars[1] -= L_ROW ? 1 : 2;
            __syncthreads();
        }
        SDRF_TICK(5);   // removal: supports + delete rows
        // ---- 5. refresh the curvature of the dirty edges ----------------------------------------------
        const int nd = min(dirty_count, S.dirty_cap);
        if (dirty_count > S.dirty_cap) {
            if (tid == 0) sh.status = DCR_SDRF_ARENA_FULL;
            __syncthreads();
            break;
        }
        for (int t = tid; t < nd; t += SDRF_THREADS) {
            const int a = S.dirty[2 * t], b = S.dirty[2 * t + 1];
            const int s = edge_slot(g, a, b);
            if (s >= 0 && atomicExch(&S.flag[s], 1) == 0) S.work[atomicAdd(&work_count, 1)] = s;
        }
        __syncthreads();
        const int nwk = work_count;
        for (int t = warp; t < nwk; t += SDRF_WARPS) {
            const int s = S.work[t];
            const int a = S.owner[s], b = S.col[s];
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

// the kernels of the loop flavour that runs DCR_SDRF_MODE_* `mode`
struct LoopKernels {
    decltype(&sdrf_init_curvature_kernel<LOOP_BFC>) init;
    decltype(&sdrf_loop_kernel<LOOP_BFC>) single;
    decltype(&sdrf_batch_loop_kernel<LOOP_BFC>) batch;
};
static LoopKernels loop_kernels(int mode) {
    switch (mode) {
    case DCR_SDRF_MODE_BFC:
        return {sdrf_init_curvature_kernel<LOOP_BFC>, sdrf_loop_kernel<LOOP_BFC>, sdrf_batch_loop_kernel<LOOP_BFC>};
    case DCR_SDRF_MODE_BFC_DIRECTED:
        return {sdrf_init_curvature_kernel<LOOP_DIRECTED>, sdrf_loop_kernel<LOOP_DIRECTED>,
                sdrf_batch_loop_kernel<LOOP_DIRECTED>};
    default:
        return {sdrf_init_curvature_kernel<LOOP_CLASSICAL>, sdrf_loop_kernel<LOOP_CLASSICAL>,
                sdrf_batch_loop_kernel<LOOP_CLASSICAL>};
    }
}

// ------------------------------------------------------------------------------------------------------------
// export
// ------------------------------------------------------------------------------------------------------------
// with_self: row lengths of the INSERTION-ORDER rows (a node that lists itself has one entry more)
__global__ void sdrf_export_rowptr_kernel(SdrfDev S, int32_t* rowptr, int with_self) {
    __shared__ Reduce red;
    // single CTA: chunked exclusive scan of rlen
    const int n = S.n;
    const int L = (n + SDRF_THREADS - 1) / SDRF_THREADS;
    const int lo = min(n, (int)threadIdx.x * L), hi = min(n, lo + L);
    long long s = 0;
    for (int v = lo; v < hi; ++v) s += S.rlen[v] + (with_self ? S.selfl[v] : 0);
    long long total;
    long long off = block_exscan_ll(s, &total, &red);
    for (int v = lo; v < hi; ++v) { rowptr[v] = (int32_t)off; off += S.rlen[v] + (with_self ? S.selfl[v] : 0); }
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
__global__ void sdrf_copy_pending_kernel(const double* pend, double* out, long long n) {
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x)
        out[t] = pend[t];
}

}  // namespace dcr

using namespace dcr;

struct dcr_sdrf {
    SdrfDev dev;
    void* slab;           // one allocation backing every array
    int mode;             // DCR_SDRF_MODE_*
    int64_t n_self;       // nodes that list themselves (self-loops of G)
};

template <class T>
static T* carve(char*& p, size_t count) {
    T* out = (T*)p;
    p += (count * sizeof(T) + 255) / 256 * 256;
    return out;
}

// rows [0,n): rowptr/order (neighbours, or successors in the directed mode); rows [n,2n): in_rowptr/in_order
// (predecessors, directed mode only)
static int sdrf_create_impl(int n, int mode, const int32_t* rowptr_host, const int32_t* order_host,
                            const int32_t* in_rowptr_host, const int32_t* in_order_host, int64_t max_additions,
                            dcr_sdrf** out) {
    if (n <= 0 || !rowptr_host || !out) { set_error("dcr_sdrf_create: bad arguments"); return 1; }
    if (mode < DCR_SDRF_MODE_BFC || mode > DCR_SDRF_MODE_HAANTJES) { set_error("dcr_sdrf_create: unknown mode"); return 1; }
    const bool directed = mode == DCR_SDRF_MODE_BFC_DIRECTED;
    if (directed && !in_rowptr_host) { set_error("dcr_sdrf_create: the directed mode needs the predecessor lists"); return 1; }
    const int rows = directed ? 2 * n : n;
    int64_t nnz = rowptr_host[n];             // (entries of the insertion-order lists; self entries are subtracted below)
    if (directed && in_rowptr_host[n] != nnz) { set_error("dcr_sdrf_create: successor / predecessor lists disagree"); return 1; }
    auto row_len = [&](int r) { return r < n ? rowptr_host[r + 1] - rowptr_host[r] : in_rowptr_host[r - n + 1] - in_rowptr_host[r - n]; };
    auto row_src = [&](int r) { return r < n ? order_host + rowptr_host[r] : in_order_host + in_rowptr_host[r - n]; };
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
            if (hits > 1) { set_error("dcr_sdrf_create: node %d lists itself more than once", me); return 1; }
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
    if (cap_total > 0x7ffffff0LL) { set_error("dcr_sdrf_create: graph too large for a 32-bit arena"); return 1; }
    std::vector<int32_t> col(sum_cap, 0), ord(sum_cap, 0), owner(sum_cap, -1);
    nnz -= n_self;                            // (directed: successor entries; the predecessor rows mirror them)
    for (int v = 0; v < rows; ++v) {
        const int len = rlen[v];
        const int32_t* src = row_src(v);
        const int self = v < n ? v : v - n;
        int filled = 0;
        for (int t = 0; t < len + selfl[v]; ++t) {
            if (src[t] < 0 || src[t] >= n || (src[t] == self && !selfl[v])) { set_error("dcr_sdrf_create: bad neighbour id"); return 1; }
            ord[rstart[v] + t] = src[t];
            if (src[t] == self) continue;
            col[rstart[v] + filled] = src[t];
            owner[rstart[v] + filled] = v;
            ++filled;
        }
        std::sort(col.begin() + rstart[v], col.begin() + rstart[v] + len);
        for (int t = 1; t < len; ++t)
            if (col[rstart[v] + t] == col[rstart[v] + t - 1]) { set_error("dcr_sdrf_create: duplicate neighbour"); return 1; }
    }
    if (directed) {   // the predecessor rows must be the transpose of the successor rows
        for (int v = 0; v < n; ++v)
            if (selfl[v] != selfl[n + v]) { set_error("dcr_sdrf_create: successor / predecessor lists disagree"); return 1; }
        for (int v = 0; v < n; ++v)
            for (int t = 0; t < rlen[v]; ++t) {
                const int w = col[rstart[v] + t];
                const int32_t* b = col.data() + rstart[n + w];
                if (!std::binary_search(b, b + rlen[n + w], v)) {
                    set_error("dcr_sdrf_create: successor / predecessor lists disagree");
                    return 1;
                }
            }
    }
    dcr_sdrf* s = new dcr_sdrf();
    s->mode = mode;
    s->n_self = n_self;
    SdrfDev& D = s->dev;
    D.n = n;
    D.ctype = mode >= DCR_SDRF_MODE_1D ? mode - DCR_SDRF_MODE_1D : 0;
    D.cap_total = (int)cap_total;
    const int64_t row_cap_max = (int64_t)d1 + max_additions + 2;
    D.row_cap_max = (int)std::min<int64_t>(row_cap_max, 0x7ffffff0LL);
    // candidate matrix: (deg x + 1)(deg y + 1) <= the product of the two longest rows after all additions
    D.imp_cap = std::min<int64_t>(((int64_t)d1 + max_additions + 2) * ((int64_t)d2 + max_additions + 2), (int64_t)1 << 28);
    // dirty pairs of one iteration: two toggles, each at most the entries at four rows + the closing edges
    D.dirty_cap = (int)std::min<int64_t>(4 * (nnz + 2 * max_additions) + 4096, 0x3ffffff0LL);
    size_t bytes = 0;
    auto add = [&](size_t count, size_t elem) { bytes += (count * elem + 255) / 256 * 256; };
    add(rows, 4); add(rows, 4); add(rows, 4); add(rows, 4);  // rstart rlen rcap selfl
    for (int i = 0; i < 6; ++i) add(cap_total, 4);           // col ord supp c32 owner flag
    add(8, 4);                                               // scalars
    for (int i = 0; i < 4; ++i) add(D.row_cap_max, 4);       // base1 base2 posI posJ
    add(D.imp_cap, 4); add(D.imp_cap, 8);                    // imp, pend
    add((size_t)2 * D.dirty_cap, 4); add(D.dirty_cap, 4);    // dirty, work
    add(D.row_cap_max, 4);                                   // wlist
    cudaError_t e = cudaMalloc(&s->slab, bytes);
    if (e != cudaSuccess) { delete s; return cuda_fail(e, "cudaMalloc(sdrf slab)", __FILE__, __LINE__); }
    char* p = (char*)s->slab;
    D.rstart = carve<int32_t>(p, rows); D.rlen = carve<int32_t>(p, rows); D.rcap = carve<int32_t>(p, rows);
    D.selfl = carve<int32_t>(p, rows);
    D.col = carve<int32_t>(p, cap_total); D.ord = carve<int32_t>(p, cap_total);
    D.supp = carve<int32_t>(p, cap_total); D.c32 = carve<float>(p, cap_total);
    D.owner = carve<int32_t>(p, cap_total); D.flag = carve<int32_t>(p, cap_total);
    D.scalars = carve<int32_t>(p, 8);
    D.base1 = carve<int32_t>(p, D.row_cap_max); D.base2 = carve<int32_t>(p, D.row_cap_max);
    D.posI = carve<int32_t>(p, D.row_cap_max); D.posJ = carve<int32_t>(p, D.row_cap_max);
    D.imp = carve<uint32_t>(p, D.imp_cap); D.pend = carve<double>(p, D.imp_cap);
    D.dirty = carve<int32_t>(p, (size_t)2 * D.dirty_cap); D.work = carve<int32_t>(p, D.dirty_cap);
    D.wlist = carve<int32_t>(p, D.row_cap_max);

    auto fail = [&](cudaError_t err, const char* what) {
        cudaFree(s->slab);
        delete s;
        return cuda_fail(err, what, __FILE__, __LINE__);
    };
#define SDRF_TRY(call) do { cudaError_t e2 = (call); if (e2 != cudaSuccess) return fail(e2, #call); } while (0)
    SDRF_TRY(cudaMemcpy(D.rstart, rstart.data(), rows * 4, cudaMemcpyHostToDevice));
    SDRF_TRY(cudaMemcpy(D.rlen, rlen.data(), rows * 4, cudaMemcpyHostToDevice));
    SDRF_TRY(cudaMemcpy(D.rcap, rcap.data(), rows * 4, cudaMemcpyHostToDevice));
    SDRF_TRY(cudaMemcpy(D.selfl, selfl.data(), rows * 4, cudaMemcpyHostToDevice));
    SDRF_TRY(cudaMemset(D.owner, 0xff, cap_total * 4));
    SDRF_TRY(cudaMemset(D.flag, 0, cap_total * 4));
    SDRF_TRY(cudaMemset(D.supp, 0, cap_total * 4));
    SDRF_TRY(cudaMemset(D.c32, 0, cap_total * 4));
    if (sum_cap > 0) {
        SDRF_TRY(cudaMemcpy(D.col, col.data(), sum_cap * 4, cudaMemcpyHostToDevice));
        SDRF_TRY(cudaMemcpy(D.ord, ord.data(), sum_cap * 4, cudaMemcpyHostToDevice));
        SDRF_TRY(cudaMemcpy(D.owner, owner.data(), sum_cap * 4, cudaMemcpyHostToDevice));
    }
    int32_t scal[8] = {(int32_t)sum_cap, (int32_t)nnz, 0, 0, 0, 0, 0, 0};
    SDRF_TRY(cudaMemcpy(D.scalars, scal, sizeof(scal), cudaMemcpyHostToDevice));
    if (sum_cap > 0) {
        const int ctas = (int)std::min<int64_t>((sum_cap + 7) / 8, (int64_t)sm_count() * 8);
        if (!directed) sdrf_init_support_kernel<<<ctas, 256>>>(D, (int)sum_cap);
        loop_kernels(mode).init<<<ctas, 256>>>(D, (int)sum_cap);
        SDRF_TRY(cudaGetLastError());
    }
    SDRF_TRY(cudaDeviceSynchronize());
#undef SDRF_TRY
    *out = s;
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
    cudaFree(s->slab);
    delete s;
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
