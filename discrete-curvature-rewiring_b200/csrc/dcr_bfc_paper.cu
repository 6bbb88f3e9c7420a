// dcr_bfc_paper.cu — paper-flavour Balanced Forman curvature over a sorted CSR (the headline kernel).
//
// Takes over bfc_edge / bfc (curvature/bfc_naive.py:7-40, :43-52).  Per undirected edge (i,j), with
//   M_i = N(i) \ N(j) \ {j},  M_j = N(j) \ N(i) \ {i}            (the "pure" neighbours of each endpoint)
// the reference's sets are
//   triangles = N(i) ∩ N(j)                                                   (:25)
//   squares_1 = {k in M_i : N(k) ∩ M_j != {}},  squares_2 mirrored            (:26-29)
//   gamma     = max over squares of |N(k) ∩ M_j| resp. |N(m) ∩ M_i|           (:36-37; the "-1" removes i / j)
// i.e. everything is a function of cnt(m) = |N(m) ∩ M_i| for m in M_j and cnt(k) = |N(k) ∩ M_j| for k in M_i.
//
// Mapping to the GPU.  (a,b) = (i,j) or (j,i): b is the endpoint whose 2-hop lists are CHEAPER to stream
// (smaller S_b - d_a); a is the TESTED endpoint.  Edges are grouped by their tested endpoint (device counting sort),
// so that the membership structures of N(a) are built once per group and READ-ONLY afterwards.  The edge classes
// below decide which kernel takes an edge:
//   * ONE WARP PER EDGE for most edges.  For d_a <= 128 the table is private to the warp and kept while consecutive
//     edges share a (paper_light_warp_kernel); above that the CTA of a group kernel builds one structure for a run of
//     edges of the same a and its warps pull edges from a shared counter (warp_edge).  The warp streams the lists
//     N(m), m a pure neighbour of b, 32 heads at a time (warp_chunk): long lists one by one, the short ones as ONE flat
//     stream whose owner arithmetic lives in the lanes' registers — no per-element search loop, no shared-memory
//     prefix arrays.  An element k is a bipartite edge (m,k) iff it is in N(a) (filter, then exact test), is not b and
//     is not a common neighbour (an exact set of T = N(a) ∩ N(b), or a mark in the d_a <= 128 table).  Matches bump
//     the list's counter (-> cnt(m)) and a match hash keyed by k (-> cnt(k)): #squares and gamma of BOTH endpoints
//     from one scan.  A warp whose match hash fills up leaves the edge to its CTA, which retries it at the end of the
//     run (cta_edge_retry: the CTA-wide hash, then a hash in global memory).
//   * COOPERATIVE edges (streams too long for one warp; hub–hub edges reach 2.5e5 streamed entries): one CTA of a
//     group kernel per edge (cta_edge), drained first; the longest are SPLIT into parts that different CTAs process.
//   * hashed mode, d_a > 16384: the CTA-team kernel (paper_edge_kernel), one 1024-thread CTA per edge, its table of
//     N(a) and slot counters in global memory, the CTA-wide flat stream cut into equal warp slices.
// Global traffic is at most the algorithmic gather of SURVEY.md §8d (which charges BOTH sides' 2-hop lists): the
// two endpoint lists once and the cheaper side's 2-hop lists once per edge.  The CSR of the benchmark graphs is
// L2-resident, so the kernel is bound by instruction issue / L1 gathers / shared-memory probes, not by DRAM.
// Grids are persistent (multiples of the SM count) and pull work from global counters.
#include <algorithm>
#include <mutex>
#include <stdlib.h>

#include "dcr_comm.cuh"

namespace dcr {

constexpr uint32_t EMPTY = 0xffffffffu;
constexpr uint32_t KEYMASK = 0x3fffffffu;
// Edge classes.  d_a = degree of the TESTED endpoint (the one whose neighbour set goes into the membership structure).
// Hashed mode (n > DENSE_MAX_N, or forced): a hashed bitmap in front of a key-only open-addressing table.
//   L0  d_a <= 128, stream <= COOP_L0    paper_light_warp_kernel: warp per edge, warp-private 256-slot table
//   G1  d_a <= 1024, stream <= COOP_G    paper_group_kernel: CTA-shared 2048-slot table, 8 warps, warp per edge
//   G2  d_a <= 16384, stream <= COOP_G   paper_group_kernel: CTA-shared 32768-slot table, 16 warps, warp per edge
//   C1 / C2  the longer streams          the group kernels of G1 / G2 (C1 also takes the long streams of L0), one CTA
//                                        per edge, drained FIRST
//   X   d_a > 16384, any stream          paper_edge_kernel: 1024-thread CTA team, table and 32-bit counters in global
//                                        memory (L2)
// Dense mode (n <= DENSE_MAX_N): L0 as above; every other edge is G1 or C1, and ONE group kernel takes both, its
// membership structure an exact bitmap over all node ids in shared memory — no table, no false positives, any degree.
// G2, C2 and X stay empty.
// In both modes an edge that a group kernel's warp cannot finish (its match hash fills up, or more than TRI_DEFER
// triangles) is retried by the warp's CTA with the CTA-wide hash, and if that fills up too, with a hash in global
// memory sized for the largest degree.
enum { CL_L0 = 0, CL_G1, CL_G2, CL_C1, CL_C2, CL_X, N_CLASSES };   // C1 / C2: the cooperative edges of G1 / G2
constexpr int CLASS_DA0 = 128, CLASS_DA1 = 1024, CLASS_DA2 = 16384;
#ifndef DCR_COOP_L0
#define DCR_COOP_L0 16384
#endif
#ifndef DCR_COOP_G
#define DCR_COOP_G 16384
#endif
// stream length above which an edge is cooperative (one CTA per edge; L0 vertices hand such edges to C1).  Measured on
// the arxiv shape at 1/1 and 1/8 of the edges per call: finer items (8192 / 4096) lose at both sizes — the CTA path
// costs more per element than the warp path.
constexpr long long COOP_L0 = DCR_COOP_L0, COOP_G = DCR_COOP_G;
// Round 2: with the long streams drained first (runs, L0 range) a warp can take longer streams without holding the tail
// of a LARGE pass: 24576 saves 3 % at 1.17 M edges per call (3.77 -> 3.65 ms) but costs 8 % at 1/8 of them, where a
// 24576-entry stream (0.25 ms on one warp) is a third of the pass — so the threshold follows the size of the call.
#ifndef DCR_COOP_BIG
#define DCR_COOP_BIG 24576
#endif
constexpr long long COOP_BIG = DCR_COOP_BIG, COOP_BIG_MIN_EDGES = 800000;
// Inside the range of one tested endpoint the light edges are ordered by size bucket, heaviest first (stream > 2048,
// > 512, the rest): warps that pull edges of a run from a shared counter then finish together.  Slot 0 of a vertex
// counts its cooperative edges: they form a second group of the vertex, in the cooperative class of its degree.
constexpr int N_SLOTS = 4;
// SPLIT edges: a stream beyond SPLIT_STREAM entries (hub–hub edges; a handful per graph, but each would occupy one CTA
// for longer than the rest of the pass takes) is cut by head ranges into parts of about SPLIT_PART entries that
// different CTAs process as independent work items; per-list results add up, the per-neighbour match counts meet in
// ONE hash in global memory per split edge, and the part that finishes last collects it and writes the result.
#ifndef DCR_SPLIT_STREAM
#define DCR_SPLIT_STREAM 98304
#endif
constexpr long long SPLIT_STREAM = DCR_SPLIT_STREAM, SPLIT_PART = 16384;
constexpr int MAX_SPLIT = 2048, MAX_PARTS = 32;
constexpr size_t SHASH_WORDS = (size_t)32 << 20;      // pool of the split edges' match hashes (128 MiB per kernel)
constexpr int SPLIT_HASH_CAP = 8192;                  // largest hash of a split edge (an edge that fills it is redone by one CTA)
struct SplitEdge {            // one per split edge, in the scratch buffer (zeroed with the plan)
    uint32_t t;               // local edge index
    int parts;                // number of parts
    int first_item;           // index of its first work item
    int tri, sq_b, g_b;       // accumulated over the parts
    int n_distinct;           // of the global hash
    int parts_done;
    int overflow;             // some part found the hash full
    uint32_t hash_off, hash_cap;   // its match hash inside the pool: 2*hash_cap words at word offset hash_off
};
constexpr long long SIZE_B1 = 2048, SIZE_B2 = 512;
// A group (all edges with the same tested endpoint) of a group class is cut into R = ceil(count / RUN_EDGES) runs;
// the edge with rank s in the size order goes to run s mod R, so EVERY run holds the same mix — heaviest first,
// lightest last — and the warps of a CTA that pull its edges from a shared counter finish together.
#ifndef DCR_RUN_EDGES
#define DCR_RUN_EDGES 64
#endif
constexpr int RUN_EDGES = DCR_RUN_EDGES;
__host__ __device__ inline int run_table_of(int cls) { return cls == CL_G2 ? 1 : 0; }
__host__ __device__ inline int coop_class_of(int cls) { return cls == CL_G2 ? CL_C2 : CL_C1; }
// Class X (CTA-team kernel): BIG_THREADS threads, one head of N(vb) per thread and round; its stream state is
// pre[BIG_THREADS+1] | beg[BIG_THREADS] | cnt[BIG_THREADS] (+ padding) in shared memory.
constexpr int BIG_THREADS = 1024, BIG_STREAM_INTS = 3 * BIG_THREADS + 8;
// Membership pre-filter: a hashed bitmap of N(va) (bit index = node id mod B).  Almost every streamed element is NOT
// a neighbour of va, and the bitmap says so with one shared-memory load and no loop; only the few elements whose bit
// is set (true members + d_a/B false positives) go on to the exact hash probe.
constexpr int GLOBAL_BITS = 1048576;
#ifndef DCR_UNROLL
#define DCR_UNROLL 4
#endif
constexpr int UNROLL = DCR_UNROLL;
// light path geometry
#ifndef DCR_L0_CTAS
#define DCR_L0_CTAS 5
#endif
#ifndef DCR_G1_CTAS
#define DCR_G1_CTAS 4
#endif
#ifndef DCR_L0_GRAB
#define DCR_L0_GRAB 4
#endif
#ifndef DCR_FLAT_UNROLL
#define DCR_FLAT_UNROLL 2
#endif
#ifndef DCR_LONG_LIST
#define DCR_LONG_LIST 64
#endif
constexpr int LONG_LIST = DCR_LONG_LIST;     // lists at least this long are streamed one at a time by the whole warp
#ifndef DCR_L0_BITS
#define DCR_L0_BITS 8192
#endif
constexpr int L0_SLOTS = 256, L0_BITS = DCR_L0_BITS, L0_WARPS = 8, L0_CTAS_PER_SM = DCR_L0_CTAS;
constexpr int G1_SLOTS = 2048, G1_BITS = 32768, G1_CAP = 512, G1_WARPS = 8, G1_CTAS_PER_SM = DCR_G1_CTAS;
constexpr int G2_SLOTS = 32768, G2_BITS = 131072, G2_CAP = 256, G2_WARPS = 16;
// dense mode: exact bitmap of N(va) over all node ids; 8 warps and >= 4 CTAs per SM while n <= DENSE_MAX_N
#ifndef DCR_GD_CTAS
#define DCR_GD_CTAS 4
#endif
#ifndef DCR_GD_WARPS
#define DCR_GD_WARPS 8
#endif
constexpr int GD_CAP = 256, GD_WARPS = DCR_GD_WARPS, GD_CTAS_PER_SM = DCR_GD_CTAS, DENSE_MAX_N = 262144;
// per-warp scratch (ints): beg[32] | len[32] | lcnt[64] (short lists by compacted rank, long lists at 32 + head lane) |
// n_distinct + pad
constexpr int WS_BEG = 0, WS_LEN = 32, WS_LCNT = 64, WS_NDIST = 128, WSTATE_INTS = 132;
// Candidate queue of a warp.  A streamed element that passes the membership filter is NOT examined on the spot (that
// code ran with one or two lanes active and was 16-22 % of all issued instructions): the lanes that hold candidates
// append (key, list) to the warp's queue with a ballot/popc compaction, and the queue is drained 32 candidates per
// pass with every lane busy — exact membership, triangle test, match counting.  It is drained when it holds
// Q_FLUSH entries and at the end of a chunk of heads / a slice, so it never holds more than Q_FLUSH - 1 + one
// window of elements.
constexpr int Q_FLUSH = 32, Q_CAP = Q_FLUSH + 32 * (DCR_UNROLL > DCR_FLAT_UNROLL ? DCR_UNROLL : DCR_FLAT_UNROLL);
constexpr int Q_WORDS = 2 * Q_CAP;
// Common neighbours T = N(va) ∩ N(vb) must not count as matches, and they are FREQUENT in the stream of a hub–hub
// edge (hubs are each other's neighbours), so membership in T has to be exact and on chip: an open-addressing set of T
// — TB_WORDS slots in the warp's scratch on the warp path (edges with |T| > TRI_DEFER go to the CTA path), sized for
// |T| on the CTA path (shared memory up to TSET_WORDS slots, this CTA's region of global memory beyond).  The d_a <=
// 128 kernel marks the slots of T in its table of N(va) instead.
constexpr int TB_WORDS = 64;
constexpr int TRI_DEFER = 32;                // light edges with more triangles go to the CTA path

struct PaperPlan {           // lives at the head of the scratch buffer
    unsigned int grouped[N_CLASSES + 1];         // [c] = #edges of class c
    unsigned int group_cursor[N_CLASSES];        // range reservation inside the classes
    unsigned int class_begin[N_CLASSES + 1];
    unsigned int next[N_CLASSES + 1];            // work-stealing counters
    unsigned int n_runs[2];                      // run tables of the group classes (G1, G2): the LIGHT runs, filled from the back
    unsigned int n_runs_heavy[2];                // ... and the HEAVY runs, filled from the front and drained first
    unsigned int coop_tier[2][4], coop_cur[2][4];   // cooperative edges of C1 / C2 by size tier (largest first): counts, cursors
    unsigned long long light_stream[2];          // streamed entries / 64 of the light edges of G1 / G2
    unsigned int l0_heavy, l0_heavy_cursor, l0_heavy_next;   // L0 edges with a stream > SIZE_B1: first in the class range, drained first
    unsigned int n_split[2], split_items[2], split_next[2];   // split edges of the kernels of G1 / G2
    unsigned long long shash_used[2];            // words of the hash pools handed out
    SplitEdge split[2][MAX_SPLIT];
};

struct PaperArgs {
    const int32_t* rowptr;
    const int32_t* colidx;
    const int32_t* esrc;
    const int32_t* edst;
    int64_t e_first, e_stride, count;  // this call handles edges e = e_first + t*e_stride, t in [0,count)
    int32_t* out_tri;
    int32_t* out_sq_i;
    int32_t* out_sq_j;
    int32_t* out_gamma;
    double* out_bfc;
    PaperPlan* plan;
    const int64_t* node_s;
    uint8_t* bucket;       // [count] class of local edge t (BUCKET_TRIVIAL: nothing to do)
    uint32_t* order;       // [count] local indices t, class by class, grouped by tested endpoint inside a class
    uint32_t* ova;         // [count] tested endpoint of order[pos]
    uint32_t* va_cnt;      // [N_SLOTS][n] #edges per (cooperative | size bucket, tested endpoint); then: rank offset inside the group
    uint32_t* va_cur;      // [N_SLOTS][n] fill cursors
    uint32_t* grp;         // [5][n] (start, count) of the vertex's light group and of its cooperative group in `order`, #runs
    uint2* runs;           // [2][max_runs] (first position, length) of the runs of the group classes
    uint32_t max_runs;
    int group_ctas;        // CTAs of a group kernel (run sizing)
    long long coop;        // stream length above which an edge is cooperative for THIS call (>= COOP_L0 / COOP_G)
    int n;
    int dense;             // 1: n is small enough for an exact bitmap of N(va) in shared memory (classes L0 + G1 only)
    uint32_t* gtables;     // class-X tables in global memory: gslots keys + gslots slot counters per CTA
    uint32_t gslots;
    uint32_t* ghash;       // last-resort match hashes in global memory: 2*ghash_cap words per CTA of a group kernel
    uint32_t ghash_cap;
    uint32_t* gtri;        // the CTA path's triangle sets that do not fit shared memory: ghash_cap words per CTA of a group kernel
    uint32_t* shash;       // [2][SHASH_WORDS] pools of the split edges' match hashes (the used part is zeroed per call)
    uint32_t* split_item;  // [2][MAX_SPLIT * MAX_PARTS] work item -> split edge << 8 | part
};

__device__ __forceinline__ uint32_t hash_slot(uint32_t key, int shift) { return (key * 2654435761u) >> shift; }

// slot of `key` in the class-X table, or -1.  The table lives in global memory and is filled with L2 atomics by
// other warps of the CTA, so it is read with ld.global.cg (L2) — an L1 line fetched during the build phase may be stale.
__device__ __forceinline__ int probe_slot(const uint32_t* tab, uint32_t mask, int shift, uint32_t key, uint32_t& val) {
    uint32_t h = hash_slot(key, shift);
    while (true) {
        const uint32_t v = __ldcg(tab + h);
        if (v == EMPTY) return -1;
        if ((v & KEYMASK) == key) { val = v; return (int)h; }
        h = (h + 1) & mask;
    }
}

// insert key with `tag`, or OR the tag into an existing entry; returns true if the key was already present
__device__ __forceinline__ bool insert_or_tag(uint32_t* tab, uint32_t mask, int shift, uint32_t key, uint32_t tag) {
    uint32_t h = hash_slot(key, shift);
    const uint32_t val = key | (tag << 30);
    while (true) {
        uint32_t v = __ldcg(tab + h);
        if (v == EMPTY) {
            v = atomicCAS(&tab[h], EMPTY, val);
            if (v == EMPTY) return false;
        }
        if ((v & KEYMASK) == key) {
            atomicOr(&tab[h], tag << 30);
            return true;
        }
        h = (h + 1) & mask;
    }
}

// ------------------------------------------------------------------------------------------------------------
// planning kernels: S_v, per-edge class/bucket, bucket offsets, order
// ------------------------------------------------------------------------------------------------------------
// S_v = sum of the degrees of v's neighbours (the two row offsets of a neighbour share a sector).
// 32 vertices per 256-thread CTA.  Rows of up to 64 entries: eight lanes per vertex (the average degree of the benchmark
// graphs is 14-76: a warp per vertex leaves most lanes idle); rows of up to 2048 entries: one warp; longer rows (hubs: a
// single warp would walk 6893 entries for 100 us after the rest of the kernel is done): the whole CTA.
__global__ void __launch_bounds__(256) node_s_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                                     int n, int64_t* __restrict__ node_s) {
    __shared__ long long s_part[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, sub = tid & 7;
    const int v0 = blockIdx.x * 32;
    auto row_sum = [&](int b, int e, int first, int step) {
        long long s = 0;
        for (int p = b + first; p < e; p += step) {
            const int k = colidx[p];
            s += rowptr[k + 1] - rowptr[k];
        }
        return s;
    };
    {
        const int v = v0 + (tid >> 3);
        long long s = 0;
        bool mine = false;
        if (v < n) {
            const int b = rowptr[v], e = rowptr[v + 1];
            mine = e - b <= 64;
            if (mine) s = row_sum(b, e, sub, 8);
        }
#pragma unroll
        for (int o = 4; o; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
        if (mine && sub == 0) node_s[v] = s;
    }
    for (int q = warp; q < 32; q += 8) {
        const int v = v0 + q;
        if (v >= n) break;
        const int b = rowptr[v], e = rowptr[v + 1];
        if (e - b <= 64 || e - b > 2048) continue;
        long long s = row_sum(b, e, lane, 32);
#pragma unroll
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
        if (lane == 0) node_s[v] = s;
    }
    for (int q = 0; q < 32; ++q) {
        const int v = v0 + q;
        if (v >= n) break;
        const int b = rowptr[v], e = rowptr[v + 1];
        if (e - b <= 2048) continue;                      // (block-uniform)
        long long s = row_sum(b, e, tid, 256);
#pragma unroll
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
        __syncthreads();
        if (lane == 0) s_part[warp] = s;
        __syncthreads();
        if (tid == 0) {
            long long t = 0;
            for (int w = 0; w < 8; ++w) t += s_part[w];
            node_s[v] = t;
        }
    }
}

constexpr int BUCKET_TRIVIAL = 255, BUCKET_SPLIT = 254;

__device__ __forceinline__ int degree_class(int da, int dense) {
    if (dense) return da <= CLASS_DA0 ? CL_L0 : CL_G1;       // the dense group kernel takes any degree
    return da <= CLASS_DA0 ? CL_L0 : (da <= CLASS_DA1 ? CL_G1 : (da <= CLASS_DA2 ? CL_G2 : CL_X));
}

// (tested endpoint, its degree, the other degree, stream size) of an edge, and where the plan puts it
struct EdgeRole { int va, da, db, cls, slot; long long stream; };
__device__ __forceinline__ EdgeRole edge_role(const PaperArgs& a, int i, int j, int di, int dj) {
    const long long ca = a.node_s[j] - di, cb = a.node_s[i] - dj;     // 2-hop entries behind j / behind i
    const bool swapped = cb < ca;                                      // stream i's side, test j
    EdgeRole r;
    r.va = swapped ? j : i;
    r.da = swapped ? dj : di;
    r.db = swapped ? di : dj;
    r.stream = swapped ? cb : ca;
    r.cls = degree_class(r.da, a.dense);
    r.slot = r.stream > SIZE_B1 ? 1 : (r.stream > SIZE_B2 ? 2 : 3);
    if (r.cls == CL_L0 ? r.stream > max(COOP_L0, a.coop) : (r.cls != CL_X && r.stream > max(COOP_G, a.coop))) {
        r.cls = coop_class_of(r.cls);                    // too long for one warp (L0 -> C1: the G1 kernel takes any degree below its own)
        r.slot = 0;
    }
    return r;
}

// Cooperative edges (one CTA per edge) are drained largest first: the CTA that would otherwise pull a 98304-entry
// stream last holds the kernel's tail.  Four size tiers inside the class range instead of a sort.
__device__ __forceinline__ int coop_tier_of(long long stream) {
    return stream >= 65536 ? 0 : (stream >= 40960 ? 1 : (stream >= 24576 ? 2 : 3));
}
// Light-group streams are accumulated per tested endpoint in units of RUN_UNIT entries (32-bit counters)
constexpr int RUN_UNIT_SHIFT = 6;

__global__ void __launch_bounds__(256) classify_kernel(PaperArgs a) {
    __shared__ unsigned int s_grp[N_CLASSES + 1];
    __shared__ unsigned int s_tier[2][4];
    __shared__ unsigned long long s_stream[2];
    __shared__ unsigned int s_l0h;
    if (threadIdx.x == 0) s_l0h = 0;
    if (threadIdx.x <= N_CLASSES) s_grp[threadIdx.x] = 0;
    if (threadIdx.x < 8) s_tier[threadIdx.x >> 2][threadIdx.x & 3] = 0;
    if (threadIdx.x < 2) s_stream[threadIdx.x] = 0;
    __syncthreads();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < a.count) {
        const int64_t e = a.e_first + t * a.e_stride;
        const int i = a.esrc[e], j = a.edst[e];
        const int di = a.rowptr[i + 1] - a.rowptr[i], dj = a.rowptr[j + 1] - a.rowptr[j];
        if (min(di, dj) <= 1) {  // bfc_naive.py:18-19: deg_min == 1 -> 0 (no triangle is possible either)
            a.out_tri[t] = 0; a.out_sq_i[t] = 0; a.out_sq_j[t] = 0; a.out_gamma[t] = 0; a.out_bfc[t] = 0.0;
            a.bucket[t] = BUCKET_TRIVIAL;
        } else {
            const EdgeRole r = edge_role(a, i, j, di, dj);
            bool split = false;
            if ((r.cls == CL_C1 || r.cls == CL_C2) && r.stream > SPLIT_STREAM) {
                const int k = r.cls == CL_C2 ? 1 : 0;
                // distinct matched neighbours <= d_a: a hash of >= 2*d_a slots never passes its 3/4 fill limit
                const uint32_t cap = 1u << (32 - __clz(min(max(2 * r.da, 1024), SPLIT_HASH_CAP) - 1));
                const unsigned long long off = atomicAdd(&a.plan->shash_used[k], 2ull * cap);
                const unsigned int sidx = (off + 2ull * cap <= SHASH_WORDS) ? atomicAdd(&a.plan->n_split[k], 1u) : MAX_SPLIT;
                if (sidx < (unsigned)MAX_SPLIT) {        // (table or pool exhausted: an ordinary cooperative edge)
                    SplitEdge& se = a.plan->split[k][sidx];
                    se.t = (uint32_t)t;
                    se.parts = (int)min((long long)min(MAX_PARTS, r.db), (r.stream + SPLIT_PART - 1) / SPLIT_PART);
                    se.first_item = (int)atomicAdd(&a.plan->split_items[k], (unsigned)se.parts);
                    se.hash_off = (uint32_t)off;
                    se.hash_cap = cap;
                    for (int q = 0; q < se.parts; ++q)
                        a.split_item[(size_t)k * MAX_SPLIT * MAX_PARTS + se.first_item + q] = (sidx << 8) | (unsigned)q;
                    split = true;
                }
            }
            if (split) {
                a.bucket[t] = BUCKET_SPLIT;
            } else {
                a.bucket[t] = (uint8_t)r.cls;
                atomicAdd(&s_grp[r.cls], 1u);
                if (r.slot == 0) {
                    atomicAdd(&s_tier[r.cls == CL_C2 ? 1 : 0][coop_tier_of(r.stream)], 1u);
                } else {
                    atomicAdd(&a.va_cnt[(size_t)r.slot * a.n + r.va], 1u);
                    if (r.cls == CL_L0 && r.slot == 1) atomicAdd(&s_l0h, 1u);
                    if (r.cls == CL_G1 || r.cls == CL_G2) {
                        const unsigned int units = (unsigned int)(r.stream >> RUN_UNIT_SHIFT) + 1u;
                        atomicAdd(&a.va_cnt[(size_t)N_SLOTS * a.n + r.va], units);
                        atomicAdd(&s_stream[run_table_of(r.cls)], (unsigned long long)units);
                    }
                }
            }
        }
    }
    __syncthreads();
    if (threadIdx.x <= N_CLASSES && s_grp[threadIdx.x]) atomicAdd(&a.plan->grouped[threadIdx.x], s_grp[threadIdx.x]);
    if (threadIdx.x < 8 && s_tier[threadIdx.x >> 2][threadIdx.x & 3])
        atomicAdd(&a.plan->coop_tier[threadIdx.x >> 2][threadIdx.x & 3], s_tier[threadIdx.x >> 2][threadIdx.x & 3]);
    if (threadIdx.x < 2 && s_stream[threadIdx.x]) atomicAdd(&a.plan->light_stream[threadIdx.x], s_stream[threadIdx.x]);
    if (threadIdx.x == 0 && s_l0h) atomicAdd(&a.plan->l0_heavy, s_l0h);
}

// position of rank s inside a group of `cnt` edges that starts at `gstart` (see RUN_EDGES)
__device__ __forceinline__ unsigned int run_layout_pos(unsigned int gstart, unsigned int cnt, unsigned int R, unsigned int s) {
    const unsigned int q = cnt / R, rem = cnt % R;
    const unsigned int r = s % R;
    return gstart + r * q + min(r, rem) + s / R;
}
// heavy runs are appended at the front of the class's run table, light runs at its back (sum of R <= #edges < max_runs)
__device__ __forceinline__ void emit_runs(const PaperArgs& a, int cls, unsigned int gstart, unsigned int cnt, unsigned int R,
                                          bool heavy) {
    const unsigned int q = cnt / R, rem = cnt % R;
    const int tbl = run_table_of(cls);
    uint2* table = a.runs + (size_t)tbl * a.max_runs;
    const unsigned int base = atomicAdd(heavy ? &a.plan->n_runs_heavy[tbl] : &a.plan->n_runs[tbl], R);
    for (unsigned int r = 0; r < R; ++r) {
        const unsigned int at = heavy ? base + r : a.max_runs - 1u - (base + r);
        table[at] = make_uint2(gstart + r * q + min(r, rem), q + (r < rem ? 1u : 0u));
    }
}
// largest stream (in run units) one run should hold: every CTA of the group kernel gets about 8 runs' worth of the
// pass, within [64 Ki, 512 Ki] entries — a run is the unit of work stealing, and the last one pulled is the tail
__device__ __forceinline__ unsigned int run_cap_units(const PaperArgs& a, int tbl) {
    const unsigned long long per = a.plan->light_stream[tbl] / (unsigned long long)(8 * max(a.group_ctas, 1));
    return (unsigned int)min(max(per, (unsigned long long)(65536 >> RUN_UNIT_SHIFT)), (unsigned long long)(524288 >> RUN_UNIT_SHIFT));
}

// Every vertex that is the tested endpoint of edges reserves a contiguous range of `order` inside the class of its
// degree for its light edges and a second one inside the cooperative class for its cooperative edges.  The order of
// the ranges is irrelevant — only contiguity matters for the table reuse — so one atomicAdd per such vertex replaces
// a scan over all vertices.  Inside a light group the size buckets follow each other, heaviest first; the group
// classes also get their run table.
__global__ void __launch_bounds__(256) plan_groups_kernel(PaperArgs a) {
    // ranges are reserved per block (shared-memory counters, then ONE global atomic per class and block): one global
    // atomic per vertex would serialise ~n operations on a handful of addresses
    __shared__ unsigned int s_cnt[N_CLASSES], s_base[N_CLASSES], s_begin[N_CLASSES + 1];
    __shared__ unsigned int s_l0h_cnt, s_l0h_base;
    if (threadIdx.x < N_CLASSES) s_cnt[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_l0h_cnt = 0;
    if (threadIdx.x == 0) {                       // class ranges: every block derives them; block 0 publishes them
        unsigned int acc = 0;
        for (int c = 0; c < N_CLASSES; ++c) { s_begin[c] = acc; acc += a.plan->grouped[c]; }
        s_begin[N_CLASSES] = acc;
        if (blockIdx.x == 0)
            for (int c = 0; c <= N_CLASSES; ++c) a.plan->class_begin[c] = s_begin[c];
    }
    // zero the handed-out part of the split edges' hash pools (grid-stride; nothing for most calls)
    for (int k = 0; k < 2; ++k) {
        const size_t used = (size_t)min(a.plan->shash_used[k], (unsigned long long)SHASH_WORDS);
        uint4* pz = (uint4*)(a.shash + (size_t)k * SHASH_WORDS);
        for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < used / 4; q += (size_t)gridDim.x * blockDim.x)
            pz[q] = make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int c[N_SLOTS] = {0, 0, 0, 0}, own = 0, own_off = 0, heavy = 0, heavy_off = 0;
    int cls = 0;
    if (v < a.n) {
        cls = degree_class(a.rowptr[v + 1] - a.rowptr[v], a.dense);
#pragma unroll
        for (int q = 0; q < N_SLOTS; ++q) {
            c[q] = a.va_cnt[(size_t)q * a.n + v];
            if (q > 0) {
                if (cls == CL_L0 && q == 1) {               // L0: the heaviest bucket forms a group of its own (see below)
                    a.va_cnt[(size_t)q * a.n + v] = 0;
                    heavy = c[q];
                } else {
                    a.va_cnt[(size_t)q * a.n + v] = own;    // rank offset of the bucket inside the light group
                    own += c[q];
                }
            }
        }
        a.va_cnt[v] = 0;
        if (own) own_off = atomicAdd(&s_cnt[cls], own);
        if (heavy) heavy_off = atomicAdd(&s_l0h_cnt, heavy);
    }
    __syncthreads();
    // The class range of L0 starts with ALL its heavy edges (stream > SIZE_B1, grouped by tested endpoint), then the rest:
    // the warps of the L0 kernel pull the long streams first, one at a time, so that no warp is left with a 16384-entry
    // stream (150 us) when the others run out of work.
    if (threadIdx.x < N_CLASSES && s_cnt[threadIdx.x])
        s_base[threadIdx.x] = s_begin[threadIdx.x] + (threadIdx.x == CL_L0 ? a.plan->l0_heavy : 0u) +
                              atomicAdd(&a.plan->group_cursor[threadIdx.x], s_cnt[threadIdx.x]);
    if (threadIdx.x == 0 && s_l0h_cnt) s_l0h_base = s_begin[CL_L0] + atomicAdd(&a.plan->l0_heavy_cursor, s_l0h_cnt);
    __syncthreads();
    if (heavy) {
        a.grp[(size_t)2 * a.n + v] = s_l0h_base + heavy_off;
        a.grp[(size_t)3 * a.n + v] = heavy;
    }
    if (own) {
        const unsigned int gstart = s_base[cls] + own_off;
        a.grp[v] = gstart;
        a.grp[(size_t)a.n + v] = own;
        if (cls == CL_G1 || cls == CL_G2) {
            // runs by edge count AND by stream: 64 edges of 16384 entries each would hold one CTA for a millisecond
            const unsigned int units = a.va_cnt[(size_t)N_SLOTS * a.n + v], cap = run_cap_units(a, run_table_of(cls));
            unsigned int R = max((own + RUN_EDGES - 1) / RUN_EDGES, (units + cap - 1) / cap);
            R = max(1u, min(R, own));
            a.grp[(size_t)4 * a.n + v] = R;
            emit_runs(a, cls, gstart, own, R, /*heavy=*/(unsigned long long)units * 4ull >= (unsigned long long)cap * R);
        }
    }
}

__global__ void __launch_bounds__(256) order_kernel(PaperArgs a) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.count) return;
    const int b = a.bucket[t];
    if (b == BUCKET_TRIVIAL || b == BUCKET_SPLIT) return;
    const int64_t e = a.e_first + t * a.e_stride;
    const int i = a.esrc[e], j = a.edst[e];
    const int di = a.rowptr[i + 1] - a.rowptr[i], dj = a.rowptr[j + 1] - a.rowptr[j];
    const EdgeRole r = edge_role(a, i, j, di, dj);
    unsigned int pos;
    if (r.slot == 0) {            // cooperative edge: by size tier inside the class range, largest first
        const int k = r.cls == CL_C2 ? 1 : 0, tier = coop_tier_of(r.stream);
        unsigned int base = a.plan->class_begin[r.cls];
        for (int q = 0; q < tier; ++q) base += a.plan->coop_tier[k][q];
        pos = base + atomicAdd(&a.plan->coop_cur[k][tier], 1u);
    } else {
        const size_t slot = (size_t)r.slot * a.n + r.va;
        const unsigned int s = a.va_cnt[slot] + atomicAdd(&a.va_cur[slot], 1u);
        const bool l0_heavy = r.cls == CL_L0 && r.slot == 1;
        const unsigned int gstart = a.grp[(l0_heavy ? (size_t)2 * a.n : 0) + r.va], cnt = a.grp[(size_t)a.n + r.va];
        pos = (r.cls == CL_G1 || r.cls == CL_G2) ? run_layout_pos(gstart, cnt, a.grp[(size_t)4 * a.n + r.va], s) : gstart + s;
    }
    a.order[pos] = (uint32_t)t;
    a.ova[pos] = (uint32_t)r.va;
}

// where a class kernel finds its work: the class's range of `order`
struct WorkSource { const uint32_t* order; unsigned int count; unsigned int* next; };
__device__ __forceinline__ WorkSource work_source(const PaperArgs& a, int cls) {
    WorkSource w;
    w.order = a.order + a.plan->class_begin[cls];
    w.count = a.plan->class_begin[cls + 1] - a.plan->class_begin[cls];
    w.next = &a.plan->next[cls];
    return w;
}

// The flat stream: `pre` = exclusive prefix sums of the list lengths (pre[l+1]-pre[l] = length of list l), `beg` =
// first CSR slot of each list, `lcnt` = per-list match counters, all in shared memory.  This warp handles the flat
// elements [f_begin, f_end) in windows of 32*UNROLL; lane f%32 takes element f.  `lw` = a list index with
// pre[lw] <= f_begin.  Windows that lie inside one list (most elements belong to long lists) take a fast path with
// no per-element owner search.  An element first meets the bitmap filter `bm`; only if its bit is set the exact
// probe runs.  A match (key present with tag 1, and not vb itself — the table holds all of N(va)) bumps the list's
// counter and the matched key's 32-bit slot counter `cnt[h]`.
__device__ __forceinline__ void flat_scan(const int32_t* __restrict__ colidx, const uint32_t* tab, uint32_t* cnt,
                                          uint32_t mask, int shift, const uint32_t* bm, const int* pre,
                                          const int* beg, int* lcnt, int lw, int f_begin, int f_end, int lane, int vb) {
    constexpr uint32_t bmask = (uint32_t)GLOBAL_BITS - 1u;
    for (int F = f_begin; F < f_end; F += 32 * UNROLL) {
        while (pre[lw + 1] <= F) ++lw;                       // warp-uniform
        const int win = min(32 * UNROLL, f_end - F);
        int k[UNROLL], lu[UNROLL];
        if (pre[lw + 1] - F >= win) {                        // the whole window lies inside list lw
            const int32_t* src = colidx + beg[lw] + (F - pre[lw]);
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const int idx = 32 * u + lane;
                k[u] = idx < win ? src[idx] : -1;
                lu[u] = lw;
            }
        } else {
            int l = lw;
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const int f = F + 32 * u + lane;
                k[u] = -1;
                lu[u] = 0;
                if (f < f_end) {
                    while (pre[l + 1] <= f) ++l;             // monotone in f: amortised O(1)
                    lu[u] = l;
                    k[u] = colidx[beg[l] + (f - pre[l])];
                }
            }
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            // vb itself sits in every streamed list (m in N(vb)) and in the table (vb in N(va)): dropping it BEFORE the
            // filter keeps the exact probe off the common path
            const uint32_t kk = (uint32_t)k[u];
            if (k[u] >= 0 && k[u] != vb && ((bm[(kk & bmask) >> 5] >> (kk & 31u)) & 1u)) {
                uint32_t v;
                const int h = probe_slot(tab, mask, shift, kk, v);
                if (h >= 0 && (v >> 30) == 1u) {
                    atomicAdd(&lcnt[lu[u]], 1);
                    atomicAdd(&cnt[h], 1u);
                }
            }
        }
    }
}

// (begin, length) of the neighbour list of head m if m is a PURE neighbour of vb (not va, not in the table), else (0,0)
__device__ __forceinline__ void pure_head(const PaperArgs& a, const uint32_t* tab, uint32_t mask, int shift, int m,
                                          int va, int& b, int& d) {
    b = 0;
    d = 0;
    uint32_t v;
    if (m != va && probe_slot(tab, mask, shift, (uint32_t)m, v) < 0) {
        b = a.rowptr[m];
        d = a.rowptr[m + 1] - b;
    }
}

// CTA team: BIG_THREADS heads per round, one per thread; the CTA-wide flat stream is cut into equal contiguous ranges,
// one per warp, so every warp streams the same number of elements whatever the list-length distribution (a hub's
// list next to twenty short ones does not serialise).  `cs` = pre[BIG_THREADS+1] | beg[BIG_THREADS] | cnt[BIG_THREADS].
__device__ __forceinline__ void scan_cta(const PaperArgs& a, const uint32_t* tab, uint32_t* cnt, uint32_t mask, int shift,
                                         const uint32_t* bm, int list_begin, int list_len, int va, int vb, int* cs,
                                         int* s_warp_tot, int& sq, int& gmax) {
    constexpr int NW = BIG_THREADS / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int* pre = cs;                      // [BIG_THREADS + 1]
    int* beg = cs + BIG_THREADS + 1;    // [BIG_THREADS]
    int* lcnt = beg + BIG_THREADS;      // [BIG_THREADS]
    for (int h0 = 0; h0 < list_len; h0 += BIG_THREADS) {
        const int nh = min(BIG_THREADS, list_len - h0);
        int b = 0, d = 0;
        if (tid < nh) pure_head(a, tab, mask, shift, a.colidx[list_begin + h0 + tid], va, b, d);
        beg[tid] = b;
        lcnt[tid] = 0;
        int inc = d;                              // exclusive scan of `d` over the CTA
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(FULL, inc, o);
            if (lane >= o) inc += up;
        }
        if (lane == 31) s_warp_tot[warp] = inc;
        __syncthreads();
        int off = inc - d;
        for (int w = 0; w < warp; ++w) off += s_warp_tot[w];
        pre[tid] = off;
        off += d;
        if (tid == BIG_THREADS - 1) pre[BIG_THREADS] = off;
        __syncthreads();
        const int total = pre[BIG_THREADS];
        if (total > 0) {
            const int per_warp = ((total + NW * 32 - 1) / (NW * 32)) * 32;
            const int f_begin = warp * per_warp, f_end = min(total, f_begin + per_warp);
            if (f_begin < f_end) {
                int lo = 0, hi = BIG_THREADS;      // first l with pre[l+1] > f_begin (warp-uniform search)
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (pre[mid + 1] <= f_begin) lo = mid + 1; else hi = mid;
                }
                flat_scan(a.colidx, tab, cnt, mask, shift, bm, pre, beg, lcnt, lo, f_begin, f_end, lane, vb);
            }
            __syncthreads();
            if (tid < nh) {
                const int c = lcnt[tid];
                sq += c > 0;
                gmax = max(gmax, c);
            }
        }
        __syncthreads();
    }
}

// CTA-team kernel (class X of hashed mode: d_a > 16384, beyond the shared-memory tables): the CTA is the team of one
// edge at a time.  The table of N(va) (gslots keys, tag in bits 30-31) and its 32-bit slot counters (gslots more words)
// live in this CTA's region of `gtables` in global memory (L2); the bitmap filter and the stream state in shared memory.
__global__ void __launch_bounds__(BIG_THREADS, 1)
paper_edge_kernel(PaperArgs a, int cls) {
    constexpr int NWARPS = BIG_THREADS / 32;
    constexpr uint32_t bmask = (uint32_t)GLOBAL_BITS - 1u;
    extern __shared__ uint32_t smem_dyn[];
    __shared__ unsigned int s_idx;
    __shared__ int s_warp_tot[NWARPS];
    __shared__ int s_red[5];  // tri, sq(lists), g(lists), sq(slots), g(slots)

    const int tid = threadIdx.x, lane = tid & 31;
    // shared-memory carve-up: [stream state][bitmap filter]
    int* st = (int*)smem_dyn;
    uint32_t* bm = smem_dyn + BIG_STREAM_INTS;
    uint32_t* tab = a.gtables + (size_t)blockIdx.x * a.gslots * 2;
    uint32_t* cnt = tab + a.gslots;
    const WorkSource ws = work_source(a, cls);
    const unsigned int cnum = ws.count;
    // edges per work-stealing step: a run of one va, usually — but never so long that the CTAs run out of steps
    const unsigned int GRAB = min(16u, max(1u, cnum / (gridDim.x * 8u)));

    int cur_va = -1;                 // vertex whose neighbour set is in the table (re-used across edges)
    uint32_t slots = 0, mask = 0;
    int shift = 0;
    while (true) {
        if (threadIdx.x == 0) s_idx = atomicAdd(ws.next, GRAB);
        __syncthreads();
        const unsigned int idx0 = s_idx;
        if (idx0 >= cnum) break;
        for (unsigned int q = 0; q < GRAB && idx0 + q < cnum; ++q) {
            if (threadIdx.x == 0) s_red[0] = s_red[1] = s_red[2] = s_red[3] = s_red[4] = 0;
            __syncthreads();
            const uint32_t t = ws.order[idx0 + q];
            const int64_t e = a.e_first + (int64_t)t * a.e_stride;
            const int i = a.esrc[e], j = a.edst[e];
            const int di = a.rowptr[i + 1] - a.rowptr[i], dj = a.rowptr[j + 1] - a.rowptr[j];
            // (va, vb): vb = endpoint whose 2-hop lists are streamed (the cheaper side), va = the tested side
            const bool swapped = (a.node_s[i] - dj) < (a.node_s[j] - di);
            const int va = swapped ? j : i, vb = swapped ? i : j;
            const int sa = a.rowptr[va], da = swapped ? dj : di;
            const int sb = a.rowptr[vb], db = swapped ? di : dj;

            if (va != cur_va) {
                // table of N(va), every key with tag 1: power of two >= 8*d_a (load factor <= 1/8 keeps probe
                // chains short and uniform across the lanes of a warp), capped by the CTA's region
                const int lg = min(32 - __clz(max(8 * da, 64) - 1), 31 - __clz(a.gslots));
                slots = 1u << lg;
                mask = slots - 1;
                shift = 32 - lg;
                for (uint32_t s = tid; s < slots; s += BIG_THREADS) tab[s] = EMPTY;
                for (uint32_t s = tid; s < slots; s += BIG_THREADS) cnt[s] = 0u;
                for (uint32_t s = tid; s < (uint32_t)GLOBAL_BITS / 32; s += BIG_THREADS) bm[s] = 0u;
                __syncthreads();
                for (int p = tid; p < da; p += BIG_THREADS) {
                    const uint32_t k = (uint32_t)a.colidx[sa + p];
                    insert_or_tag(tab, mask, shift, k, 1u);
                    atomicOr(&bm[(k & bmask) >> 5], 1u << (k & 31u));
                }
                __syncthreads();
                cur_va = va;
            }
            // common neighbours: heads of N(vb) found in the table get bit 31 (tag 3: never a match, never a head)
            int tri = 0;
            for (int p = tid; p < db; p += BIG_THREADS) {
                const int m = a.colidx[sb + p];
                uint32_t v;
                const int h = (m == va) ? -1 : probe_slot(tab, mask, shift, (uint32_t)m, v);
                if (h >= 0) {
                    atomicOr(&tab[h], 2u << 30);
                    ++tri;
                }
            }
            tri = warp_sum(tri);
            if (lane == 0 && tri) atomicAdd(&s_red[0], tri);
            __syncthreads();

            // the scan: lists of the pure neighbours of vb, matches against the pure neighbours of va
            int sqL = 0, gL = 0, sqS = 0, gS = 0;
            scan_cta(a, tab, cnt, mask, shift, bm, sb, db, va, vb, st, s_warp_tot, sqL, gL);
            sqL = warp_sum(sqL);
            gL = warp_max(gL);
            if (lane == 0 && sqL) { atomicAdd(&s_red[1], sqL); atomicMax(&s_red[2], gL); }
            __syncthreads();
            sqL = s_red[1]; gL = s_red[2]; tri = s_red[0];
            // the collect: slot counters of the pure neighbours of va -> squares at va (empty iff the scan found
            // nothing).  Walks N(va) (d_a probes) instead of sweeping the table and zeroes the counters it reads,
            // so the table is clean for the next edge of the same va.
            if (sqL > 0) {
                for (int p = tid; p < da; p += BIG_THREADS) {
                    const int k = a.colidx[sa + p];
                    uint32_t v;
                    const int h = probe_slot(tab, mask, shift, (uint32_t)k, v);
                    if (h >= 0 && (v >> 30) == 1u) {
                        const int c = (int)__ldcg(cnt + (uint32_t)h);
                        if (c > 0) {
                            ++sqS;
                            gS = max(gS, c);
                            cnt[h] = 0u;
                        }
                    }
                }
                sqS = warp_sum(sqS);
                gS = warp_max(gS);
                if (lane == 0 && sqS) { atomicAdd(&s_red[3], sqS); atomicMax(&s_red[4], gS); }
                __syncthreads();
                sqS = s_red[3]; gS = s_red[4];
            }
            if (tid == 0) {
                const int sq_i = swapped ? sqL : sqS, sq_j = swapped ? sqS : sqL;
                const int gamma = (sqL > 0 && sqS > 0) ? max(gL, gS) : 0;
                a.out_tri[t] = tri;
                a.out_sq_i[t] = sq_i;
                a.out_sq_j[t] = sq_j;
                a.out_gamma[t] = gamma;      // the fp64 value is computed by paper_value_kernel (one thread per edge)
            }
            // undo the common-neighbour marks so the table is N(va) with tag 1 again
            if (tri > 0) {
                for (int p = tid; p < db; p += BIG_THREADS) {
                    const int m = a.colidx[sb + p];
                    uint32_t v;
                    const int h = (m == va) ? -1 : probe_slot(tab, mask, shift, (uint32_t)m, v);
                    if (h >= 0) atomicAnd(&tab[h], 0x7fffffffu);
                }
            }
            __syncthreads();  // table / s_red reuse
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// warp-granular edges over READ-ONLY membership structures of N(va)
// ------------------------------------------------------------------------------------------------------------
__host__ __device__ constexpr int ilog2_c(int v) { return v <= 1 ? 0 : 1 + ilog2_c(v >> 1); }

// slot of `key` in a key-only table, or -1
__device__ __forceinline__ int ro_probe(const uint32_t* tab, uint32_t mask, int shift, uint32_t key) {
    uint32_t h = hash_slot(key, shift);
    while (true) {
        const uint32_t v = tab[h];
        if (v == key) return (int)h;
        if (v == EMPTY) return -1;
        h = (h + 1) & mask;
    }
}
__device__ __forceinline__ void ro_insert(uint32_t* tab, uint32_t mask, int shift, uint32_t key) {
    uint32_t h = hash_slot(key, shift);
    while (true) {
        const uint32_t v = atomicCAS(&tab[h], EMPTY, key);
        if (v == EMPTY || v == key) return;
        h = (h + 1) & mask;
    }
}
__device__ __forceinline__ bool bitmap_test(const uint32_t* bm, uint32_t bmask, uint32_t k) {
    return (bm[(k & bmask) >> 5] >> (k & 31u)) & 1u;
}

// Table geometry for a tested endpoint of degree d_a: power of two >= 2*d_a slots (>= 64), key-only.
template <int MAX_SLOTS>
__device__ __forceinline__ void ro_geometry(int da, uint32_t& mask, int& shift) {
    const int lg = min(32 - __clz(max(2 * da, 64) - 1), ilog2_c(MAX_SLOTS));
    mask = (1u << lg) - 1u;
    shift = 32 - lg;
}

// Membership in N(va).  DENSE: an exact bitmap over all node ids in shared memory (one load, no probe) — used when
// n bits fit beside the rest of the CTA state.  Otherwise: hashed bitmap pre-filter + key-only open-addressing table.
template <bool DENSE>
struct Member {
    const uint32_t* tab;
    const uint32_t* bm;
    uint32_t mask, bmask;
    int shift;
    __device__ __forceinline__ bool maybe(uint32_t k) const {      // cheap necessary condition (exact when DENSE)
        return DENSE ? ((bm[k >> 5] >> (k & 31u)) & 1u) : bitmap_test(bm, bmask, k);
    }
    __device__ __forceinline__ uint32_t word(uint32_t k) const { return DENSE ? bm[k >> 5] : bm[(k & bmask) >> 5]; }
    __device__ __forceinline__ bool confirm(uint32_t k) const {    // after maybe(k)
        return DENSE ? true : (ro_probe(tab, mask, shift, k) >= 0);
    }
    __device__ __forceinline__ bool has(uint32_t k) const { return maybe(k) && confirm(k); }
};

// One out-of-line copy per kernel: the candidate path is cold next to the streaming loops, and the group kernels had
// outgrown the instruction cache (stall_no_instructions was the top stall reason with everything inlined).
__device__ __noinline__ bool match_hash_add(uint32_t* mh, int* n_distinct, uint32_t cap, int shift, uint32_t k) {
    const uint32_t key = k + 1u;
    uint32_t p = (key * 0x9E3779B1u) >> shift;
    for (uint32_t tries = 0; tries < cap; ++tries) {
        uint32_t v = *(volatile uint32_t*)(mh + p);
        if (v == 0u) {
            if (*(volatile int*)n_distinct >= (int)(cap / 4 * 3)) return false;
            v = atomicCAS(&mh[p], 0u, key);
            if (v == 0u) atomicAdd(n_distinct, 1);
        }
        if (v == 0u || v == key) {
            atomicAdd(&mh[cap + p], 1u);
            return true;
        }
        p = (p + 1) & (cap - 1);
    }
    return false;
}

// Match hash: keys[cap] (node id + 1) | counts[cap], cap a power of two; lives in shared memory (per warp, or the
// per-warp hashes of a CTA taken together) or, as a last resort, in global memory.
struct MatchHash {
    uint32_t* mh;
    int* n_distinct;
    uint32_t cap;
    int shift;            // 32 - log2(cap)
    __device__ __forceinline__ void init(uint32_t* p, int* nd, uint32_t c) {
        mh = p; n_distinct = nd; cap = c; shift = __clz(c) + 1;
    }
    // false when the hash is (nearly) full
    __device__ __forceinline__ bool add(uint32_t k) { return match_hash_add(mh, n_distinct, cap, shift, k); }
    // (#distinct keys, largest count) of this thread's share of the hash; clears what it reads
    __device__ __forceinline__ void collect(int first, int stride, int& sq_a, int& g_a) {
        for (uint32_t p = first; p < cap; p += stride) {
            if (*(volatile uint32_t*)(mh + p)) {
                ++sq_a;
                g_a = max(g_a, (int)*(volatile uint32_t*)(mh + cap + p));
                mh[p] = 0u;
                mh[cap + p] = 0u;
            }
        }
    }
};

// Everything a warp needs to test streamed elements of one edge (va tested, vb streamed) against the CTA-level or
// warp-level structures of the group kernels: membership in N(va), the structure that answers "k in T", the match
// hash, the warp's candidate queue and the per-list match counters the queue entries point into.
template <bool DENSE>
struct EdgeCtx {
    const int32_t* __restrict__ colidx;
    Member<DENSE> mem;
    const uint32_t* tb;      // exact open-addressing set of T (per warp in shared memory, or the CTA's: shared / global)
    uint32_t tb_mask;        // slots - 1 (0: the empty set)
    int tb_shift;            // 32 - log2(slots)
    bool tb_global;          // the set lives in global memory (filled with L2 atomics: read with ld.global.cg)
    MatchHash hash;
    uint32_t* q;             // candidate queue: (key, list) pairs, or key | list << 24 in one word when DENSE (n <= 2^18)
    int qn;                  // its length (warp-uniform)
    static constexpr int Q_ENTRY_WORDS = DENSE ? 1 : 2;
    __device__ __forceinline__ void q_store(int pos, uint32_t k, uint32_t list) {
        if (DENSE) q[pos] = k | (list << 24);
        else ((uint2*)q)[pos] = make_uint2(k, list);
    }
    __device__ __forceinline__ void q_load(int pos, uint32_t& k, uint32_t& list) const {
        if (DENSE) { const uint32_t v = q[pos]; k = v & 0xffffffu; list = v >> 24; }
        else { const uint2 v = ((const uint2*)q)[pos]; k = v.x; list = v.y; }
    }
    int* lcnt;               // per-list match counters
    int va, vb, sb, db;
    bool ovf;
    __device__ __forceinline__ bool in_triangle(uint32_t kk) const {
        uint32_t h = ((kk * 2654435761u) >> tb_shift) & tb_mask;
        while (true) {
            const uint32_t v = tb_global ? __ldcg(tb + h) : tb[h];
            if (v == kk) return true;
            if (v == EMPTY) return false;
            h = (h + 1) & tb_mask;
        }
    }
    // k in N(m), m a pure neighbour of vb: is (m,k) an edge of the bipartite graph M_b – M_a?  hit() is the per-element
    // filter of the streaming loops (one shared-memory load); handle() runs on queued candidates, 32 per pass.
    __device__ __forceinline__ uint32_t word(int k) const { return mem.word((uint32_t)k); }
    __device__ __forceinline__ void handle(uint32_t kk, uint32_t list) {
        if ((int)kk != vb && mem.confirm(kk) && !in_triangle(kk)) {     // k in N(va) \ {vb} and not a common neighbour
            if (!hash.add(kk)) ovf = true;
            atomicAdd(&lcnt[list], 1);
        }
    }
};
__device__ __forceinline__ void tri_set_insert(uint32_t* ts, uint32_t mask, int shift, uint32_t kk) {
    uint32_t h = ((kk * 2654435761u) >> shift) & mask;
    while (true) {
        const uint32_t v = atomicCAS(&ts[h], EMPTY, kk);
        if (v == EMPTY || v == kk) return;
        h = (h + 1) & mask;
    }
}

// Append this window's candidates (bit u of hm: element k[u] of this lane passed the filter) to the warp's queue: one
// ballot per element row, lanes that hold a candidate of the row store it behind the candidates of the lower lanes.
template <class Ctx, int N>
__device__ __forceinline__ void q_push(Ctx& cx, uint32_t hm, const int (&k)[N], const int (&own)[N], int lane) {
    const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
    for (int u = 0; u < N; ++u) {
        const bool mine = (hm >> u) & 1u;
        const uint32_t b = __ballot_sync(FULL, mine);
        if (b) {
            if (mine) cx.q_store(cx.qn + __popc(b & lt), (uint32_t)k[u], (uint32_t)own[u]);
            cx.qn += __popc(b);
        }
    }
}
template <class Ctx>
__device__ __forceinline__ void q_flush(Ctx& cx, int lane) {
    __syncwarp();
    for (int q = lane; q < cx.qn; q += 32) {
        uint32_t k, list;
        cx.q_load(q, k, list);
        cx.handle(k, list);
    }
    cx.qn = 0;
    __syncwarp();
}

// The filter of one window: bit u of the result says that element k[u] of this lane may be a match.  The filter word of
// element u is rotated so that the element's bit lands on bit u (one funnel shift) and merged with one and-or; the
// streamed endpoint itself — it sits in every streamed list and in N(va) — is dropped here.
template <class Ctx, int N>
__device__ __forceinline__ uint32_t filter_window(const Ctx& cx, const int (&k)[N]) {
    uint32_t w[N];
#pragma unroll
    for (int u = 0; u < N; ++u) w[u] = cx.word(k[u]);
    uint32_t hm = 0;
#pragma unroll
    for (int u = 0; u < N; ++u) hm |= __funnelshift_r(w[u], w[u], (uint32_t)k[u] - (uint32_t)u) & (1u << u);
#pragma unroll
    for (int u = 0; u < N; ++u) if (k[u] == cx.vb) hm &= ~(1u << u);
    return hm;
}

// `len` consecutive entries of ONE neighbour list, streamed by the whole warp (p already includes the lane offset);
// candidates go to the queue with `owner` as their list.  Full windows carry no bounds test at all; lanes past the
// end of the last window test va, which is never a member of N(va).
template <class Ctx>
__device__ __forceinline__ void stream_list(Ctx& cx, const int32_t* __restrict__ p, int len, int owner, int lane) {
    int own[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) own[u] = owner;
    const int full = len & ~(32 * UNROLL - 1);
    for (int F = 0; F < full; F += 32 * UNROLL) {           // all loads of a window are in flight before the first test
        int k[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) k[u] = __ldg(p + F + 32 * u);
        const uint32_t hm = filter_window(cx, k);
        if (__any_sync(FULL, hm != 0u)) {
            q_push(cx, hm, k, own, lane);
            if (cx.qn >= Q_FLUSH) q_flush(cx, lane);
        }
    }
    const int rem = len - full;
    if (rem) {
        int k[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) k[u] = (32 * u + lane < rem) ? __ldg(p + full + 32 * u) : cx.va;
        const uint32_t hm = filter_window(cx, k);
        if (__any_sync(FULL, hm != 0u)) {
            q_push(cx, hm, k, own, lane);
            if (cx.qn >= Q_FLUSH) q_flush(cx, lane);
        }
    }
}
// (out-of-line copies work on a register copy of the context: through the reference every store to shared memory
//  would force the context's fields to be re-read from the caller's stack frame)
template <class Ctx>
__device__ __noinline__ void stream_list_call(Ctx& cx_ref, const int32_t* __restrict__ p, int len, int owner, int lane) {
    Ctx cx = cx_ref;
    stream_list(cx, p, len, owner, lane);
    cx_ref.qn = cx.qn;
    cx_ref.ovf = cx.ovf;
}

// One chunk of 32 heads of N(vb) by one warp; lane l holds head l of the chunk: (mb, md) = (begin, length) of its
// neighbour list if the head is a PURE neighbour of vb, else (0, 0).  Lists of at least LONG_LIST entries are streamed
// one at a time by the whole warp (no ownership arithmetic at all); the shorter ones form ONE flat stream — the
// (begin - prefix) of each list lives in a lane's register, the owner of flat element f is found with one warp-wide
// OR-reduction of the "a list starts here" bits plus a popc, its data come through one shuffle.  Candidates of both
// go through the queue; the chunk ends with the queue drained and the per-list counters folded into the lane-partial
// sq_b (#lists with a match) and g_b (largest per-list count).
template <class Ctx>
__device__ __forceinline__ void warp_chunk(Ctx& cx, int mb, int md, int* st, int lane, int& sq_b, int& g_b) {
    const int32_t* __restrict__ colidx = cx.colidx;
    const uint32_t lm0 = __ballot_sync(FULL, md >= LONG_LIST);
    const bool shortl = md > 1 && md < LONG_LIST;               // (a list that holds only vb cannot match)
    const uint32_t pm = __ballot_sync(FULL, shortl);
    if ((lm0 | pm) == 0u) return;
    int* sbeg = st + WS_BEG;
    int* slen = st + WS_LEN;
    int* lcnt = st + WS_LCNT;
    lcnt[lane] = 0;
    lcnt[32 + lane] = 0;
    const int nl = __popc(pm);
    if (shortl) {
        const int r = __popc(pm & ((1u << lane) - 1u));
        sbeg[r] = mb;
        slen[r] = md;
    }
    __syncwarp();
    // long lists
    uint32_t lm = lm0;
    while (lm) {
        const int src = __ffs(lm) - 1;
        lm &= lm - 1;
        const int len = __shfl_sync(FULL, md, src);
        stream_list(cx, colidx + __shfl_sync(FULL, mb, src) + lane, len, 32 + src, lane);
    }
    // short lists
    if (pm) {
        const int len_l = lane < nl ? slen[lane] : 0;
        int inc = len_l;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(FULL, inc, o);
            if (lane >= o) inc += up;
        }
        const int total = __shfl_sync(FULL, inc, 31);
        const int pre_l = lane < nl ? inc - len_l : 0x3fffffff;      // flat position of the first element of list `lane`
        const int base_l = (lane < nl ? sbeg[lane] : 0) - pre_l;     // colidx index of flat element f of this list: base + f
        const uint32_t le_mask = 0xffffffffu >> (31 - lane);
        int below = 0;                                               // #lists that start before the current group
        constexpr int FU = DCR_FLAT_UNROLL;
        for (int F = 0; F < total; F += 32 * FU) {
            int k[FU], own[FU];
#pragma unroll
            for (int u = 0; u < FU; ++u) {
                const int Fu = F + 32 * u;
                const unsigned rel = (unsigned)(pre_l - Fu);
                const uint32_t starts = __reduce_or_sync(FULL, rel < 32u ? (1u << rel) : 0u);
                own[u] = (below + __popc(starts & le_mask) - 1) & 31;
                below += __popc(starts);
                const int bs = __shfl_sync(FULL, base_l, own[u]);
                const int f = Fu + lane;
                k[u] = f < total ? __ldg(colidx + bs + f) : cx.va;
            }
            const uint32_t hm = filter_window(cx, k);
            if (__any_sync(FULL, hm != 0u)) {
                q_push(cx, hm, k, own, lane);
                if (cx.qn >= Q_FLUSH) q_flush(cx, lane);
            }
        }
    }
    if (cx.qn) q_flush(cx, lane); else __syncwarp();
    const int c1 = lcnt[lane], c2 = lcnt[32 + lane];
    sq_b += (c1 > 0) + (c2 > 0);
    g_b = max(g_b, max(c1, c2));
    __syncwarp();
}

// the warp paths inline the chunk; cta_edge calls this out-of-line copy
template <class Ctx>
__device__ __noinline__ void warp_chunk_call(Ctx& cx_ref, int mb, int md, int* st, int lane, int& sq_b_ref, int& g_b_ref) {
    Ctx cx = cx_ref;
    int sq_b = sq_b_ref, g_b = g_b_ref;
    warp_chunk(cx, mb, md, st, lane, sq_b, g_b);
    sq_b_ref = sq_b;
    g_b_ref = g_b;
    cx_ref.qn = cx.qn;
    cx_ref.ovf = cx.ovf;
}

// One edge by one warp over the CTA-level membership structure (group kernels).  `st` = the warp's scratch, `tb` =
// its exact triangle set (TB_WORDS words), `mh` = its match hash (2*CAP words, all zero on entry and on exit), `q` = its
// candidate queue.  Writes the four integer fields of local edge t and returns true, or returns false when the match
// hash filled up or the edge has too many triangles for the warp's set (nothing written; the hash is clean again).
template <int CAP, bool DENSE>
__device__ __forceinline__ bool warp_edge(const PaperArgs& a, const Member<DENSE>& mem, uint32_t t, int va, int* st,
                                          uint32_t* tb, uint32_t* mh, uint32_t* q, int lane) {
    const int64_t e = a.e_first + (int64_t)t * a.e_stride;
    const int i = a.esrc[e], j = a.edst[e];
    const bool swapped = (va == j);                      // stream i's side, test j
    EdgeCtx<DENSE> cx;
    cx.colidx = a.colidx; cx.mem = mem; cx.tb = tb; cx.tb_mask = TB_WORDS - 1; cx.tb_shift = 32 - ilog2_c(TB_WORDS);
    cx.tb_global = false; cx.hash.init(mh, st + WS_NDIST, CAP);
    cx.q = q; cx.qn = 0; cx.lcnt = st + WS_LCNT;
    cx.va = va;
    cx.vb = swapped ? i : j;
    cx.sb = a.rowptr[cx.vb];
    cx.db = a.rowptr[cx.vb + 1] - cx.sb;
    cx.ovf = false;
    // pass 1 over the heads: the common neighbours (triangles).  Lane l looks at heads l, l+32, ...; whether head
    // l + 32c is in N(va) is remembered in bit c of `mbits` (heads beyond 1024 are looked up again in pass 2).
    int tri = 0;
    uint32_t mbits = 0;
    for (int p = lane, c = 0; p < cx.db; p += 32, ++c) {
        const uint32_t m = (uint32_t)a.colidx[cx.sb + p];
        const bool in = ((int)m != va && mem.has(m));
        tri += in;
        if (c < 32) mbits |= in ? (1u << c) : 0u;
    }
    tri = __reduce_add_sync(FULL, tri);
    // the warp's exact set of T holds TB_WORDS/2 keys: a richer edge goes to the CTA path
    if (tri > TRI_DEFER) return false;
    if (tri > 0) {
        for (int p = lane; p < TB_WORDS; p += 32) tb[p] = EMPTY;
        __syncwarp();
        for (int p = lane, c = 0; p < cx.db; p += 32, ++c) {
            if (c < 32 && !((mbits >> c) & 1u)) continue;
            const uint32_t m = (uint32_t)a.colidx[cx.sb + p];
            if (c < 32 || ((int)m != va && mem.has(m))) tri_set_insert(tb, TB_WORDS - 1, 32 - ilog2_c(TB_WORDS), m);
        }
    } else if (lane == 0) {
        tb[0] = EMPTY;                                   // an empty set is recognised by its first probe ...
    }
    if (tri == 0) cx.tb_mask = 0;                        // ... every key hashes to slot 0
    __syncwarp();
    // pass 2: the lists of the pure heads
    int sq_b = 0, g_b = 0;
    for (int c0 = 0, c = 0; c0 < cx.db; c0 += 32, ++c) {
        int mb = 0, md = 0;
        if (c0 + lane < cx.db) {
            const int m = a.colidx[cx.sb + c0 + lane];
            const bool in = c < 32 ? ((mbits >> c) & 1u) : mem.has((uint32_t)m);
            if (m != va && !in) {
                mb = a.rowptr[m];
                md = a.rowptr[m + 1] - mb;
            }
        }
        warp_chunk(cx, mb, md, st, lane, sq_b, g_b);
    }
    sq_b = __reduce_add_sync(FULL, sq_b);
    g_b = __reduce_max_sync(FULL, g_b);
    int sq_a = 0, g_a = 0;
    if (sq_b > 0) {                                      // the match hash is non-empty iff some list matched
        cx.hash.collect(lane, 32, sq_a, g_a);
        sq_a = __reduce_add_sync(FULL, sq_a);
        g_a = __reduce_max_sync(FULL, g_a);
        if (lane == 0) st[WS_NDIST] = 0;
    }
    const bool ovf = __any_sync(FULL, cx.ovf);
    if (lane == 0 && !ovf) {
        a.out_tri[t] = tri;
        a.out_sq_i[t] = swapped ? sq_b : sq_a;
        a.out_sq_j[t] = swapped ? sq_a : sq_b;
        a.out_gamma[t] = (sq_b > 0 && sq_a > 0) ? max(g_a, g_b) : 0;
    }
    __syncwarp();
    return !ovf;
}

// ------------------------------------------------------------------------------------------------------------
// L0 (d_a <= 128): everything private to the warp.  The key-only table of N(va) doubles as the match structure:
// `cnt[h]` belongs to the key in slot h — bit 31 marks a common neighbour (never a match), the low bits count the
// matches of the current edge — so a candidate costs ONE probe (membership, triangle test and match counter at once)
// and there is neither a triangle set nor a match hash.  At most 128 distinct keys: nothing can overflow.
// ------------------------------------------------------------------------------------------------------------
constexpr uint32_t L0_TRI = 0x80000000u;
struct L0Ctx {
    const int32_t* __restrict__ colidx;
    const uint32_t* tab;
    const uint32_t* bm;
    uint32_t* cnt;
    uint32_t mask;
    int shift;
    uint32_t* q;
    int qn;
    int* lcnt;
    int va, vb, sb, db;
    __device__ __forceinline__ void q_store(int pos, uint32_t k, uint32_t list) { ((uint2*)q)[pos] = make_uint2(k, list); }
    __device__ __forceinline__ void q_load(int pos, uint32_t& k, uint32_t& list) const {
        const uint2 v = ((const uint2*)q)[pos];
        k = v.x; list = v.y;
    }
    uint32_t bm_off;          // byte offset of this warp's filter inside the CTA's filter block (a multiple of its size)
    // one shift, one and-or, one load at a constant shared-memory base: the filters of the CTA's warps are contiguous
    // at the start of dynamic shared memory and each is a power of two long
    __device__ __forceinline__ uint32_t word(int k) const {
        extern __shared__ uint32_t smem_dyn[];
        return *(const uint32_t*)((const char*)smem_dyn + ((((uint32_t)k >> 3) & (L0_BITS / 8 - 4)) | bm_off));
    }
    __device__ __forceinline__ void handle(uint32_t kk, uint32_t list) {
        const int h = ro_probe(tab, mask, shift, kk);
        if (h >= 0 && !(*(volatile uint32_t*)(cnt + h) & L0_TRI)) {
            atomicAdd(&cnt[h], 1u);
            atomicAdd(&lcnt[list], 1);
        }
    }
};

__device__ __forceinline__ void warp_edge_l0(const PaperArgs& a, L0Ctx& cx, uint32_t t, int va, int* st, int lane) {
    const int64_t e = a.e_first + (int64_t)t * a.e_stride;
    const int i = a.esrc[e], j = a.edst[e];
    const bool swapped = (va == j);                      // stream i's side, test j
    cx.vb = swapped ? i : j;
    cx.sb = a.rowptr[cx.vb];
    cx.db = a.rowptr[cx.vb + 1] - cx.sb;
    cx.qn = 0;
    cx.va = va;
    // vb is in N(va) and in every streamed list, and never a match: its slot carries the mark of the common neighbours
    if (lane == 0) cx.cnt[ro_probe(cx.tab, cx.mask, cx.shift, (uint32_t)cx.vb)] = L0_TRI;
    // pass 1 over the heads: common neighbours get their slot marked
    int tri = 0;
    uint32_t mbits = 0;
    for (int p = lane, c = 0; p < cx.db; p += 32, ++c) {
        const uint32_t m = (uint32_t)a.colidx[cx.sb + p];
        bool in = false;
        if ((int)m != va && bitmap_test(cx.bm, L0_BITS - 1, m)) {
            const int h = ro_probe(cx.tab, cx.mask, cx.shift, m);
            if (h >= 0) { cx.cnt[h] = L0_TRI; in = true; }
        }
        tri += in;
        if (c < 32) mbits |= in ? (1u << c) : 0u;
    }
    tri = __reduce_add_sync(FULL, tri);
    __syncwarp();
    // pass 2: the lists of the pure heads
    int sq_b = 0, g_b = 0;
    for (int c0 = 0, c = 0; c0 < cx.db; c0 += 32, ++c) {
        int mb = 0, md = 0;
        if (c0 + lane < cx.db) {
            const int m = a.colidx[cx.sb + c0 + lane];
            const bool in = c < 32 ? ((mbits >> c) & 1u)
                                   : (bitmap_test(cx.bm, L0_BITS - 1, (uint32_t)m) && ro_probe(cx.tab, cx.mask, cx.shift, (uint32_t)m) >= 0);
            if (m != va && !in) {
                mb = a.rowptr[m];
                md = a.rowptr[m + 1] - mb;
            }
        }
        warp_chunk(cx, mb, md, st, lane, sq_b, g_b);
    }
    sq_b = __reduce_add_sync(FULL, sq_b);
    g_b = __reduce_max_sync(FULL, g_b);
    // the collect: one sweep over the slot counters reads the matches of va's side and leaves them all zero
    int sq_a = 0, g_a = 0;
    {
        for (uint32_t s = lane; s <= cx.mask; s += 32) {
            const uint32_t c = cx.cnt[s];
            if (c) {
                cx.cnt[s] = 0u;
                if (!(c & L0_TRI)) { ++sq_a; g_a = max(g_a, (int)c); }
            }
        }
        sq_a = __reduce_add_sync(FULL, sq_a);
        g_a = __reduce_max_sync(FULL, g_a);
    }
    if (lane == 0) {
        a.out_tri[t] = tri;
        a.out_sq_i[t] = swapped ? sq_b : sq_a;
        a.out_sq_j[t] = swapped ? sq_a : sq_b;
        a.out_gamma[t] = (sq_b > 0 && sq_a > 0) ? max(g_a, g_b) : 0;
    }
    __syncwarp();
}

// L0 kernel: warp-private table, kept while consecutive edges (sorted by tested endpoint) share va.
constexpr int L0_PER_WARP = WSTATE_INTS + Q_WORDS + 2 * L0_SLOTS;      // beside the filter
__global__ void __launch_bounds__(L0_WARPS * 32, L0_CTAS_PER_SM) paper_light_warp_kernel(PaperArgs a) {
    extern __shared__ uint32_t smem_dyn[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // [filters of the 8 warps, contiguous][per warp: scratch | queue | table | slot counters]
    uint32_t* bm = smem_dyn + warp * (L0_BITS / 32);
    uint32_t* base = smem_dyn + L0_WARPS * (L0_BITS / 32) + warp * L0_PER_WARP;
    int* st = (int*)base;
    uint32_t* tab = base + WSTATE_INTS + Q_WORDS;
    uint32_t* cnt = tab + L0_SLOTS;
    for (int p = lane; p < L0_SLOTS; p += 32) cnt[p] = 0u;
    __syncwarp();
    const WorkSource ws = work_source(a, CL_L0);
    const uint32_t* ova = a.ova + a.plan->class_begin[CL_L0];
    int cur_va = -1;
    L0Ctx cx;
    cx.colidx = a.colidx; cx.tab = tab; cx.bm = bm; cx.cnt = cnt; cx.mask = 0; cx.shift = 0;
    cx.q = base + WSTATE_INTS; cx.qn = 0; cx.lcnt = st + WS_LCNT;
    cx.bm_off = (uint32_t)warp * (L0_BITS / 8);
    const unsigned int n_heavy = a.plan->l0_heavy;       // the class range starts with the long streams: one per grab
    bool heavy_phase = n_heavy > 0;
    while (true) {
        unsigned int idx0 = 0, idx1;
        if (heavy_phase) {
            if (lane == 0) idx0 = atomicAdd(&a.plan->l0_heavy_next, 1u);
            idx0 = __shfl_sync(FULL, idx0, 0);
            if (idx0 >= n_heavy) { heavy_phase = false; continue; }
            idx1 = idx0 + 1u;
        } else {
            if (lane == 0) idx0 = atomicAdd(ws.next, (unsigned)DCR_L0_GRAB);
            idx0 = __shfl_sync(FULL, idx0, 0) + n_heavy;
            if (idx0 >= ws.count) break;
            idx1 = min(ws.count, idx0 + (unsigned)DCR_L0_GRAB);
        }
        for (unsigned int q = idx0; q < idx1; ++q) {
            const int va = (int)ova[q];
            if (va != cur_va) {
                const int sa = a.rowptr[va], da = a.rowptr[va + 1] - sa;
                ro_geometry<L0_SLOTS>(da, cx.mask, cx.shift);
                for (uint32_t s = lane; s <= cx.mask; s += 32) tab[s] = EMPTY;
                for (int s = lane; s < L0_BITS / 32; s += 32) bm[s] = 0u;
                __syncwarp();
                for (int p = lane; p < da; p += 32) {
                    const uint32_t k = (uint32_t)a.colidx[sa + p];
                    ro_insert(tab, cx.mask, cx.shift, k);
                    atomicOr(&bm[(k & (L0_BITS - 1)) >> 5], 1u << (k & 31u));
                }
                __syncwarp();
                cur_va = va;
            }
            warp_edge_l0(a, cx, ws.order[q], va, st, lane);
        }
    }
}


// One COOPERATIVE edge by the whole CTA (stream too long, too many triangles or too many distinct matches for one
// warp).  No rounds and no CTA-wide prefix sums: the warps pull CHUNKS of 32 heads from a shared counter and process
// each exactly like the warp path does (warp_chunk: long lists one at a time, short lists as one flat stream,
// candidates through the warp's queue) — the only CTA barriers are the ones around the triangle set at the start and
// the reductions at the end.  What is shared by the CTA: the exact set of T (shared memory up to TSET_WORDS slots,
// beyond that this CTA's region of `gtri` in global memory), the match hash (the per-warp hashes taken together, or a
// hash in global memory) and the BIG lists: a list of at least BIG_LIST entries (hub neighbours) would hold one warp
// long after the others ran out of chunks, so it is parked in s_big and, once the chunks are done, streamed by all
// warps in slices of BIG_SLICE entries.
// s_acc: [0] tri (this part) [1] sq_b [2] g_b [3] next chunk [4] n_distinct [5] overflow [6] sq_a [7] g_a [8] "this
// part finalises its split edge" [9] |T| [10] #big lists.  All threads call it; the caller synchronises the CTA before
// the next use of s_acc.
// (round 2: 15 % of the group kernel's stall samples sat on the barrier that ends the chunk loop — a warp whose chunk
// holds a 2000-entry list keeps the other seven waiting; parking lists from 1024 entries on and slicing them 512 at a
// time took the 1/8-range pass from 0.71 to 0.67 ms and the full pass from 3.65 to 3.63; 512 / 256 were no better)
#ifndef DCR_BIG_LIST
#define DCR_BIG_LIST 1024
#endif
#ifndef DCR_BIG_SLICE
#define DCR_BIG_SLICE 512
#endif
#ifndef DCR_MAX_BIG
#define DCR_MAX_BIG 64
#endif
constexpr int TSET_WORDS = 1024, BIG_LIST = DCR_BIG_LIST, BIG_SLICE = DCR_BIG_SLICE, MAX_BIG = DCR_MAX_BIG;
template <int NWARPS, bool DENSE>
__device__ __noinline__ void cta_edge(const PaperArgs& a, const Member<DENSE>& mem, uint32_t t, int va, int* st_all,
                                      uint32_t* tset_sh, uint32_t* hash_words, uint32_t hash_cap, uint32_t* q_all, int* s_acc,
                                      int* s_big, int part, int parts, SplitEdge* se) {
    constexpr int THREADS = NWARPS * 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int* st = st_all + warp * WSTATE_INTS;
    const int64_t e = a.e_first + (int64_t)t * a.e_stride;
    const int i = a.esrc[e], j = a.edst[e];
    const bool swapped = (va == j);
    EdgeCtx<DENSE> cx;
    cx.colidx = a.colidx; cx.mem = mem;
    cx.hash.init(hash_words, se ? &se->n_distinct : s_acc + 4, hash_cap);
    cx.q = q_all + warp * (Q_CAP * cx.Q_ENTRY_WORDS); cx.qn = 0; cx.lcnt = st + WS_LCNT;
    cx.va = va;
    cx.vb = swapped ? i : j;
    cx.sb = a.rowptr[cx.vb];
    cx.db = a.rowptr[cx.vb + 1] - cx.sb;
    cx.ovf = false;
    // a part of a split edge takes the heads [h_lo, h_hi) (the triangle set always covers all heads)
    const int h_lo = (int)((long long)cx.db * part / parts), h_hi = (int)((long long)cx.db * (part + 1) / parts);
    if (tid < 12) s_acc[tid] = 0;
    __syncthreads();
    // the common neighbours: count, then build the exact set sized for them
    int tri = 0, tri_all = 0;
    for (int p = tid; p < cx.db; p += THREADS) {
        const uint32_t m = (uint32_t)a.colidx[cx.sb + p];
        const bool in = ((int)m != va && mem.has(m));
        tri_all += in;
        tri += in && p >= h_lo && p < h_hi;
    }
    tri = __reduce_add_sync(FULL, tri);
    tri_all = __reduce_add_sync(FULL, tri_all);
    if (lane == 0 && tri_all) { atomicAdd(&s_acc[0], tri); atomicAdd(&s_acc[9], tri_all); }
    __syncthreads();
    const int n_t = s_acc[9];
    if (n_t == 0) {
        cx.tb = tset_sh; cx.tb_mask = 0; cx.tb_shift = 31; cx.tb_global = false;
        if (tid == 0) tset_sh[0] = EMPTY;
    } else {
        const int lg = max(6, 32 - __clz(2 * n_t - 1));            // >= 2 |T| slots
        const uint32_t slots = 1u << lg;
        cx.tb_global = slots > (uint32_t)TSET_WORDS;
        uint32_t* ts = cx.tb_global ? a.gtri + (size_t)blockIdx.x * a.ghash_cap : tset_sh;   // ghash_cap >= pow2(2 * max degree)
        cx.tb = ts; cx.tb_mask = slots - 1; cx.tb_shift = 32 - lg;
        for (uint32_t s = tid; s < slots; s += THREADS) ts[s] = EMPTY;
        __syncthreads();
        for (int p = tid; p < cx.db; p += THREADS) {
            const uint32_t m = (uint32_t)a.colidx[cx.sb + p];
            if ((int)m != va && mem.has(m)) tri_set_insert(ts, cx.tb_mask, cx.tb_shift, m);
        }
    }
    __syncthreads();
    // the chunks of the part's heads
    int sq_b = 0, g_b = 0;
    const int nchunks = (h_hi - h_lo + 31) >> 5;
    while (true) {
        int c = 0;
        if (lane == 0) c = atomicAdd(&s_acc[3], 1);
        c = __shfl_sync(FULL, c, 0);
        if (c >= nchunks) break;
        const int p = h_lo + 32 * c + lane;
        int mb = 0, md = 0;
        if (p < h_hi) {
            const int m = a.colidx[cx.sb + p];
            if (m != va && !mem.has((uint32_t)m)) {
                mb = a.rowptr[m];
                md = a.rowptr[m + 1] - mb;
            }
        }
        const uint32_t bigm = __ballot_sync(FULL, md >= BIG_LIST);
        if (bigm) {                                   // park the big lists (those that find no room stay with this warp)
            int slot = 0;
            if (lane == 0) slot = atomicAdd(&s_acc[10], __popc(bigm));
            slot = __shfl_sync(FULL, slot, 0) + __popc(bigm & ((1u << lane) - 1u));
            if (md >= BIG_LIST && slot < MAX_BIG) {
                s_big[slot] = mb;
                s_big[MAX_BIG + slot] = md;
                s_big[2 * MAX_BIG + slot] = 0;
                mb = 0;
                md = 0;
            }
        }
        warp_chunk_call(cx, mb, md, st, lane, sq_b, g_b);
    }
    __syncthreads();
    const int nbig = min(s_acc[10], MAX_BIG);
    if (nbig) {
        cx.lcnt = s_big + 2 * MAX_BIG;
        int before = 0;                               // slices of the earlier lists: slice q of the edge goes to warp q mod NWARPS
        for (int b = 0; b < nbig; ++b) {
            const int beg = s_big[b], len = s_big[MAX_BIG + b];
            const int ns = (len + BIG_SLICE - 1) / BIG_SLICE;
            for (int s = ((warp - before) % NWARPS + NWARPS) % NWARPS; s < ns; s += NWARPS)
                stream_list_call(cx, a.colidx + beg + s * BIG_SLICE + lane, min(BIG_SLICE, len - s * BIG_SLICE), b, lane);
            before += ns;
        }
        if (cx.qn) q_flush(cx, lane);
        __syncthreads();
        if (tid < nbig) {
            const int c = s_big[2 * MAX_BIG + tid];
            sq_b += c > 0;
            g_b = max(g_b, c);
        }
    }
    sq_b = __reduce_add_sync(FULL, sq_b);
    g_b = __reduce_max_sync(FULL, g_b);
    const bool ovf = __any_sync(FULL, cx.ovf);
    if (lane == 0) {
        if (sq_b) { atomicAdd(&s_acc[1], sq_b); atomicMax(&s_acc[2], g_b); }
        if (ovf) s_acc[5] = 1;
    }
    __syncthreads();
    int tri_out = s_acc[0], sq_b_all = s_acc[1], g_b_all = s_acc[2];
    bool finalise = true;
    if (se) {     // publish this part; the part that finishes last collects the shared hash and writes the result
        if (tid == 0) {
            atomicAdd(&se->tri, s_acc[0]);
            atomicAdd(&se->sq_b, s_acc[1]);
            atomicMax(&se->g_b, s_acc[2]);
            if (s_acc[5]) atomicOr(&se->overflow, 1);
            __threadfence();
            s_acc[8] = (atomicAdd(&se->parts_done, 1) == parts - 1);
            s_acc[5] = 0;
        }
        __syncthreads();
        finalise = s_acc[8] != 0;
        if (finalise) {
            __threadfence();
            if (tid == 0) s_acc[5] = *(volatile int*)&se->overflow;   // the caller redoes the edge on its own
            __syncthreads();
            tri_out = *(volatile int*)&se->tri;
            sq_b_all = *(volatile int*)&se->sq_b;
            g_b_all = *(volatile int*)&se->g_b;
        }
    }
    if (finalise && sq_b_all > 0) {
        int sq_a = 0, g_a = 0;
        cx.hash.collect(tid, THREADS, sq_a, g_a);
        sq_a = __reduce_add_sync(FULL, sq_a);
        g_a = __reduce_max_sync(FULL, g_a);
        if (lane == 0 && sq_a) { atomicAdd(&s_acc[6], sq_a); atomicMax(&s_acc[7], g_a); }
        __syncthreads();
    }
    if (finalise && tid == 0 && !s_acc[5]) {
        const int sa_ = s_acc[6];
        a.out_tri[t] = tri_out;
        a.out_sq_i[t] = swapped ? sq_b_all : sa_;
        a.out_sq_j[t] = swapped ? sa_ : sq_b_all;
        a.out_gamma[t] = (sq_b_all > 0 && sa_ > 0) ? max(g_b_all, s_acc[7]) : 0;
    }
}


#ifdef DCR_PAPER_TRACE
// debug: per CTA of the group kernel [t_begin, t_phase1_end, t_end, longest item ns, its (phase<<30 | index), #items]
__device__ unsigned long long g_trace[4096 * 6];
__device__ unsigned long long g_trace_cnt[8];   // [0] deferred edges [1] their stream [2] CTA-path edges that needed the big hash
__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define TRACE(...) __VA_ARGS__
#else
#define TRACE(...)
#endif

// cooperative edge with the CTA-wide shared hash; on overflow once more with this CTA's hash in global memory
// (2*ghash_cap words, ghash_cap >= 2 * max degree: it cannot fill up).  Ends with the CTA synchronised.
template <int NWARPS, int CAP, bool DENSE>
__device__ __forceinline__ void cta_edge_retry(const PaperArgs& a, const Member<DENSE>& mem, uint32_t t, int va,
                                               int* st_all, uint32_t* tset_sh, uint32_t* mh_all, uint32_t* q_all, int* s_acc,
                                               int* s_big) {
    cta_edge<NWARPS, DENSE>(a, mem, t, va, st_all, tset_sh, mh_all, NWARPS * CAP, q_all, s_acc, s_big, 0, 1, nullptr);
    __syncthreads();
    TRACE(if (threadIdx.x == 0) { atomicAdd(&g_trace_cnt[3], 1ull); if (s_acc[5]) atomicAdd(&g_trace_cnt[2], 1ull); })
    if (s_acc[5]) {
        uint32_t* gh = a.ghash + (size_t)blockIdx.x * 2 * a.ghash_cap;
        for (uint32_t p = threadIdx.x; p < 2 * a.ghash_cap; p += NWARPS * 32) gh[p] = 0u;
        __threadfence_block();
        __syncthreads();
        cta_edge<NWARPS, DENSE>(a, mem, t, va, st_all, tset_sh, gh, a.ghash_cap, q_all, s_acc, s_big, 0, 1, nullptr);
        __syncthreads();
    }
}


// (Re)build the membership structures of N(va) for the CTA; all threads; ends synchronised.  One out-of-line copy (three
// call sites in the group kernel).
template <int NWARPS, int MAX_SLOTS, bool DENSE>
__device__ __noinline__ void build_member(const PaperArgs& a, Member<DENSE>& mem, uint32_t* tab, uint32_t* bm, int bm_words,
                                          int& prev_va, int va) {
    constexpr int THREADS = NWARPS * 32;
    const int tid = threadIdx.x;
    if (prev_va == va) return;
    const int sa = a.rowptr[va], da = a.rowptr[va + 1] - sa;
    if (DENSE) {
        if (prev_va >= 0) {                        // un-set the previous endpoint's bits (no full clear)
            const int ps = a.rowptr[prev_va], pd = a.rowptr[prev_va + 1] - ps;
#pragma unroll 1
            for (int p = tid; p < pd; p += THREADS) {
                const uint32_t k = (uint32_t)a.colidx[ps + p];
                atomicAnd(&bm[k >> 5], ~(1u << (k & 31u)));
            }
        }
    } else {
        ro_geometry<MAX_SLOTS>(da, mem.mask, mem.shift);
#pragma unroll 1
        for (uint32_t s = tid; s <= mem.mask; s += THREADS) tab[s] = EMPTY;
#pragma unroll 1
        for (int s = tid; s < bm_words; s += THREADS) bm[s] = 0u;
    }
    __syncthreads();
#pragma unroll 1
    for (int p = tid; p < da; p += THREADS) {
        const uint32_t k = (uint32_t)a.colidx[sa + p];
        if (DENSE) {
            atomicOr(&bm[k >> 5], 1u << (k & 31u));
        } else {
            ro_insert(tab, mem.mask, mem.shift, k);
            atomicOr(&bm[(k & mem.bmask) >> 5], 1u << (k & 31u));
        }
    }
    prev_va = va;
    __syncthreads();
}

// Group kernel: the CTA builds the membership structures of N(va) for a run of edges with the same tested endpoint.
// The cooperative edges of the run (they come first) are processed by the whole CTA one at a time; then the warps
// pull the remaining edges — ordered by size, heaviest first — from a shared counter, one warp per edge; edges whose
// per-warp match hash filled up are retried cooperatively at the end of the run.
// DENSE: exact bitmap over all n node ids (dense_words 32-bit words); otherwise hashed bitmap + table.
template <int NWARPS, int MAX_SLOTS, int BITS, int CAP, int CTAS_PER_SM, bool DENSE>
__global__ void __launch_bounds__(NWARPS * 32, CTAS_PER_SM) paper_group_kernel(PaperArgs a, int cls, int dense_words) {
    extern __shared__ uint32_t smem_dyn[];
    __shared__ unsigned int s_idx, s_next;
    __shared__ int s_ndefer;
    __shared__ uint32_t s_defer[RUN_EDGES];
    __shared__ int s_acc[12];      // [8]: "this part finalises its split edge"
    __shared__ int s_big[3 * MAX_BIG];
    constexpr int THREADS = NWARPS * 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // [CTA-path triangle set: TSET_WORDS][per-warp triangle sets: NWARPS x TB_WORDS][match hashes: NWARPS x
    // 2*CAP][warp scratch: NWARPS x WSTATE_INTS][table (hashed only)][bitmap: hashed BITS/32 words | dense dense_words]
    uint32_t* tb_coop = smem_dyn;                          // the CTA path's exact set of T (TSET_WORDS slots)
    constexpr int tb_coop_words = TSET_WORDS;
    uint32_t* tb_all = tb_coop + tb_coop_words;
    uint32_t* mh_all = tb_all + NWARPS * TB_WORDS;
    int* st_all = (int*)(mh_all + NWARPS * 2 * CAP);
    constexpr int QW = Q_CAP * (DENSE ? 1 : 2);                      // words per warp queue
    uint32_t* q_all = (uint32_t*)(st_all + NWARPS * WSTATE_INTS);    // per-warp candidate queues (8-byte aligned: all sizes even)
    uint32_t* tab = q_all + NWARPS * QW;
    uint32_t* bm = tab + (DENSE ? 0 : MAX_SLOTS);
    const int bm_words = DENSE ? dense_words : BITS / 32;
    int* st = st_all + warp * WSTATE_INTS;
    uint32_t* tb = tb_all + warp * TB_WORDS;
    // warp-private view: keys[CAP] | counts[CAP] inside the warp's 2*CAP words; cooperative view: keys[NWARPS*CAP] |
    // counts[NWARPS*CAP] over the whole region.  Both rely on the region being all zero between edges.
    uint32_t* mh = mh_all + warp * 2 * CAP;
    for (int p = tid; p < NWARPS * 2 * CAP; p += THREADS) mh_all[p] = 0u;
    if (lane == 0) st[WS_NDIST] = 0;
    if (DENSE) {
        for (int s = tid; s < bm_words; s += THREADS) bm[s] = 0u;
    }
    const uint2* runs = a.runs + (size_t)run_table_of(cls) * a.max_runs;
    const unsigned int n_heavy = a.plan->n_runs_heavy[run_table_of(cls)];
    const unsigned int n_runs = n_heavy + a.plan->n_runs[run_table_of(cls)];   // heavy runs first, then the light ones
    const int ccls = coop_class_of(cls);
    const WorkSource cws = work_source(a, ccls);
    const uint32_t* cova = a.ova + a.plan->class_begin[ccls];
    Member<DENSE> mem;
    mem.tab = tab; mem.bm = bm; mem.bmask = BITS - 1; mem.mask = 0; mem.shift = 0;
    int prev_va = -1;
    auto build = [&](int va) { build_member<NWARPS, MAX_SLOTS, DENSE>(a, mem, tab, bm, bm_words, prev_va, va); };
    TRACE(unsigned long long tr_t0 = gtimer(), tr_long = 0, tr_id = 0, tr_n = 0;)
    // phase 0: the parts of the split edges — by far the longest streams of the pass
    {
        const int k = run_table_of(cls);
        const unsigned int items = a.plan->split_items[k];
        while (true) {
            __syncthreads();
            if (tid == 0) s_idx = atomicAdd(&a.plan->split_next[k], 1u);
            __syncthreads();
            const int item = (int)s_idx;
            if ((unsigned)item >= items) break;
            TRACE(const unsigned long long tr_a = gtimer();)
            const uint32_t code = a.split_item[(size_t)k * MAX_SPLIT * MAX_PARTS + item];
            const int sidx = (int)(code >> 8), part = (int)(code & 255u);
            SplitEdge* se = &a.plan->split[k][sidx];
            const uint32_t t = se->t;
            const int64_t e = a.e_first + (int64_t)t * a.e_stride;
            const int i = a.esrc[e], j = a.edst[e];
            const int va = edge_role(a, i, j, a.rowptr[i + 1] - a.rowptr[i], a.rowptr[j + 1] - a.rowptr[j]).va;
            build(va);
            cta_edge<NWARPS, DENSE>(a, mem, t, va, st_all, tb_coop, a.shash + (size_t)k * SHASH_WORDS + se->hash_off,
                                    se->hash_cap, q_all, s_acc, s_big, part, se->parts, se);
            __syncthreads();
            if (s_acc[8] && s_acc[5]) {                  // its hash filled up: once more, whole, with this CTA's big hash
                uint32_t* gh = a.ghash + (size_t)blockIdx.x * 2 * a.ghash_cap;
                for (uint32_t p = tid; p < 2 * a.ghash_cap; p += THREADS) gh[p] = 0u;
                __threadfence_block();
                __syncthreads();
                cta_edge<NWARPS, DENSE>(a, mem, t, va, st_all, tb_coop, gh, a.ghash_cap, q_all, s_acc, s_big, 0, 1, nullptr);
            }
            TRACE(const unsigned long long tr_d = gtimer() - tr_a; ++tr_n; if (tr_d > tr_long) { tr_long = tr_d; tr_id = (3ull << 30) | t; })
        }
    }
    // phase 1: the cooperative edges, one per work item — the heaviest work of the pass starts first
    while (true) {
        __syncthreads();                                  // s_idx reuse
        if (tid == 0) s_idx = atomicAdd(cws.next, 1u);
        __syncthreads();
        const unsigned int idx = s_idx;
        if (idx >= cws.count) break;
        TRACE(const unsigned long long tr_a = gtimer();)
        const int va = (int)cova[idx];
        build(va);
        cta_edge_retry<NWARPS, CAP, DENSE>(a, mem, cws.order[idx], va, st_all, tb_coop, mh_all, q_all, s_acc, s_big);
        TRACE(const unsigned long long tr_d = gtimer() - tr_a; ++tr_n; if (tr_d > tr_long) { tr_long = tr_d; tr_id = (1ull << 30) | cws.order[idx]; })
    }
    TRACE(const unsigned long long tr_t1 = gtimer();)
    if (lane == 0) st[WS_NDIST] = 0;                      // the cooperative stream state overlays the warp scratch
    // phase 2: runs of light edges of one tested endpoint, ordered by size; one warp per edge
    while (true) {
        __syncthreads();
        if (tid == 0) { s_idx = atomicAdd(&a.plan->next[cls], 1u); s_next = 0; s_ndefer = 0; }
        __syncthreads();
        if (s_idx >= n_runs) break;
        TRACE(const unsigned long long tr_a = gtimer();)
        const uint2 run = runs[s_idx < n_heavy ? s_idx : a.max_runs - 1u - (s_idx - n_heavy)];   // (first position in `order`, length)
        const uint32_t* ord = a.order + run.x;
        const int q_end = (int)run.y;
        const int va = (int)a.ova[run.x];
        build(va);
        while (true) {
            unsigned int my = 0;
            if (lane == 0) my = atomicAdd(&s_next, 1u);
            my = __shfl_sync(FULL, my, 0);
            if ((int)my >= q_end) break;
            const uint32_t t = ord[my];
            if (!warp_edge<CAP, DENSE>(a, mem, t, va, st, tb, mh, q_all + warp * QW, lane) && lane == 0)
                s_defer[atomicAdd(&s_ndefer, 1)] = t;     // too many triangles / distinct matches for one warp: CTA path
        }
        __syncthreads();                                  // every warp is done with the run
        const int nd = s_ndefer;
        TRACE(if (tid == 0 && nd) atomicAdd(&g_trace_cnt[0], (unsigned long long)nd);)
        for (int d = 0; d < nd; ++d)
            cta_edge_retry<NWARPS, CAP, DENSE>(a, mem, s_defer[d], va, st_all, tb_coop, mh_all, q_all, s_acc, s_big);
        if (nd > 0 && lane == 0) st[WS_NDIST] = 0;
        TRACE(const unsigned long long tr_d = gtimer() - tr_a; ++tr_n; if (tr_d > tr_long) { tr_long = tr_d; tr_id = (2ull << 30) | ((unsigned long long)nd << 20) | s_idx; })
    }
    TRACE(if (tid == 0 && blockIdx.x < 4096) { unsigned long long* r = g_trace + blockIdx.x * 6; r[0] = tr_t0; r[1] = tr_t1; r[2] = gtimer(); r[3] = tr_long; r[4] = tr_id; r[5] = tr_n; })
}

// bfc_naive.py:31-32 / :39-40 for every edge of the call, one thread per edge: the eight fp64 divisions would
// otherwise run on one lane of the edge's team.
__global__ void paper_value_kernel(PaperArgs a) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.count) return;
    const int64_t e = a.e_first + t * a.e_stride;
    const int i = a.esrc[e], j = a.edst[e];
    const int di = a.rowptr[i + 1] - a.rowptr[i], dj = a.rowptr[j + 1] - a.rowptr[j];
    if (min(di, dj) <= 1) return;      // written by classify_kernel: the int 0 of bfc_naive.py:18-19
    a.out_bfc[t] = paper_value(di, dj, a.out_tri[t], a.out_sq_i[t], a.out_sq_j[t], a.out_gamma[t]);
}

}  // namespace dcr

using namespace dcr;

static inline uint32_t next_pow2_u32(uint64_t v) {
    uint32_t p = 64;
    while (p < v) p <<= 1;
    return p;
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Membership mode: 0 = automatic (exact shared-memory bitmap up to DENSE_MAX_N nodes), 1 = force the hashed-table
// kernels (the path of graphs with more than DENSE_MAX_N nodes) — used by the parity tests to cover both paths on
// small graphs.  The initial value comes from the environment variable DCR_PAPER_MODE=hashed, read ONCE at load;
// dcr_bfc_paper_set_mode() changes it (process-wide; call it between passes, not concurrently with one).
static int g_paper_mode = []() {
    const char* m = getenv("DCR_PAPER_MODE");
    return (m && m[0] == 'h') ? 1 : 0;
}();
extern "C" int dcr_bfc_paper_set_mode(int mode) {
    const int old = g_paper_mode;
    g_paper_mode = mode ? 1 : 0;
    return old;
}
static bool use_dense_mode(int n) { return g_paper_mode == 0 && n <= DENSE_MAX_N; }

struct ScratchLayout {
    size_t plan, node_s, bucket, order, ova, va_cnt, va_cur, grp, runs, gtables, ghash, gtri, shash, split_item, zero_bytes, total;
    uint32_t max_runs;
    uint32_t gslots, ghash_cap;
    int g_ctas, group_ctas;
};

static ScratchLayout scratch_layout(int n, int max_degree, int64_t count) {
    ScratchLayout L;
    size_t off = 0;
    // plan | va_cnt | va_cur are adjacent: one memset clears the three of them
    L.plan = off; off = align_up(off + sizeof(PaperPlan), 256);
    L.va_cnt = off; off = align_up(off + (size_t)(N_SLOTS + 1) * n * sizeof(uint32_t), 256);   // + the light-group streams
    L.va_cur = off; off = align_up(off + (size_t)N_SLOTS * n * sizeof(uint32_t), 256);
    L.zero_bytes = off;
    L.node_s = off; off = align_up(off + (size_t)n * sizeof(int64_t), 256);
    L.bucket = off; off = align_up(off + (size_t)count, 256);
    L.order = off; off = align_up(off + (size_t)count * sizeof(uint32_t), 256);
    L.ova = off; off = align_up(off + (size_t)count * sizeof(uint32_t), 256);
    L.grp = off; off = align_up(off + (size_t)5 * n * sizeof(uint32_t), 256);
    // a light group of c edges is cut into at most c runs (by edge count and by stream)
    L.max_runs = (uint32_t)(count + 1);
    L.runs = off; off = align_up(off + (size_t)2 * L.max_runs * sizeof(uint2), 256);
    // tables of the CTA-team kernel (class X: tested endpoints beyond the shared-memory tables, hashed mode only)
    L.gslots = 0;
    L.g_ctas = 0;
    L.gtables = off;
    if (max_degree > CLASS_DA2 && !use_dense_mode(n)) {
        L.gslots = next_pow2_u32((uint64_t)max_degree * 4);
        L.g_ctas = sm_count();
        off = align_up(off + (size_t)L.g_ctas * L.gslots * 2 * sizeof(uint32_t), 256);   // keys + counters
    }
    // last-resort match hashes of the group kernels (one per CTA; zeroed by the CTA that needs one)
    L.ghash_cap = std::max<uint32_t>(4096u, next_pow2_u32((uint64_t)max_degree * 2));
    L.group_ctas = sm_count() * std::max(GD_CTAS_PER_SM, G1_CTAS_PER_SM);
    L.ghash = off; off = align_up(off + (size_t)L.group_ctas * 2 * L.ghash_cap * sizeof(uint32_t), 256);
    L.gtri = off; off = align_up(off + (size_t)L.group_ctas * L.ghash_cap * sizeof(uint32_t), 256);
    L.shash = off; off = align_up(off + (size_t)2 * SHASH_WORDS * sizeof(uint32_t), 256);
    L.split_item = off; off = align_up(off + (size_t)2 * MAX_SPLIT * MAX_PARTS * sizeof(uint32_t), 256);
    L.total = off;
    return L;
}

extern "C" int64_t dcr_bfc_paper_scratch_bytes(int n, int max_degree, int64_t count) {
    return (int64_t)scratch_layout(n, max_degree, count).total;
}

// per-device fork/join streams and events of the pass.  One pass at a time per device may use them: the section
// that records / waits on them is serialised by the device's mutex (two host threads driving the same device with
// different streams would otherwise re-record each other's fork event).
struct PaperAux {
    std::mutex mu;
    bool ready = false, attr_done = false;
    cudaStream_t aux[3] = {};
    cudaEvent_t fork = nullptr, join[3] = {};
};
static PaperAux g_aux[MAX_DEVICES];

static int paper_pass(const int32_t* rowptr, const int32_t* colidx, int n, int max_degree,
                      const int32_t* esrc, const int32_t* edst, int64_t e_first, int64_t e_stride,
                      int64_t count, int32_t* out_tri, int32_t* out_sq_i, int32_t* out_sq_j,
                      int32_t* out_gamma, double* out_bfc, void* scratch, int64_t scratch_bytes,
                      void* ev_edge_begin, void* ev_edge_end, void* stream, bool value_kernel) {
    if (count <= 0 || n <= 0) return 0;
    if (count > 0xfffffff0LL) { set_error("dcr_bfc_paper: more than 2^32 edges per call"); return 1; }
    if (n >= (1 << 30) - 1) { set_error("dcr_bfc_paper: node ids must fit 30 bits (table keys carry 2 tag bits)"); return 1; }
    if (max_degree > (1 << 22)) {   // 256 lists of a cooperative round are laid out as one 32-bit flat stream
        set_error("dcr_bfc_paper: max_degree %d above 2^22 is not supported", max_degree);
        return 1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const ScratchLayout L = scratch_layout(n, max_degree, count);
    if ((int64_t)L.total > scratch_bytes) {
        set_error("dcr_bfc_paper: scratch too small (%lld < %lld bytes)", (long long)scratch_bytes, (long long)L.total);
        return 1;
    }
    char* base = (char*)scratch;
    PaperArgs a;
    a.rowptr = rowptr; a.colidx = colidx; a.esrc = esrc; a.edst = edst;
    a.e_first = e_first; a.e_stride = e_stride; a.count = count;
    a.out_tri = out_tri; a.out_sq_i = out_sq_i; a.out_sq_j = out_sq_j; a.out_gamma = out_gamma; a.out_bfc = out_bfc;
    a.plan = (PaperPlan*)(base + L.plan);
    int64_t* node_s = (int64_t*)(base + L.node_s);
    a.node_s = node_s;
    a.bucket = (uint8_t*)(base + L.bucket);
    a.order = (uint32_t*)(base + L.order);
    a.ova = (uint32_t*)(base + L.ova);
    a.va_cnt = (uint32_t*)(base + L.va_cnt);
    a.va_cur = (uint32_t*)(base + L.va_cur);
    a.grp = (uint32_t*)(base + L.grp);
    a.runs = (uint2*)(base + L.runs);
    a.max_runs = L.max_runs;
    a.group_ctas = L.group_ctas;
    a.coop = count >= COOP_BIG_MIN_EDGES ? COOP_BIG : 0;
    a.n = n;
    a.dense = use_dense_mode(n) ? 1 : 0;
    a.gtables = (uint32_t*)(base + L.gtables);
    a.gslots = L.gslots;
    a.ghash = (uint32_t*)(base + L.ghash);
    a.ghash_cap = L.ghash_cap;
    a.gtri = (uint32_t*)(base + L.gtri);
    a.shash = (uint32_t*)(base + L.shash);
    a.split_item = (uint32_t*)(base + L.split_item);

    DCR_CUDA(cudaMemsetAsync(base + L.plan, 0, L.zero_bytes - L.plan, st));      // plan, va_cnt, va_cur
    node_s_kernel<<<(unsigned)((n + 31) / 32), 256, 0, st>>>(rowptr, colidx, n, node_s);
    DCR_LAUNCH_CHECK();
    const unsigned tb = (unsigned)((count + 255) / 256);
    classify_kernel<<<tb, 256, 0, st>>>(a);
    DCR_LAUNCH_CHECK();
    plan_groups_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a);     // + class ranges, + zeroing of the split hashes
    DCR_LAUNCH_CHECK();
    order_kernel<<<tb, 256, 0, st>>>(a);
    DCR_LAUNCH_CHECK();

    const int sms = sm_count();
    if (ev_edge_begin) DCR_CUDA(cudaEventRecord((cudaEvent_t)ev_edge_begin, st));
    // Persistent grids = SM count x resident CTAs per SM.
    const int dev = current_device();
    PaperAux& ax = g_aux[dev];
    std::lock_guard<std::mutex> guard(ax.mu);
    bool& attr_done = ax.attr_done;
    const int dense_words = (n + 63) / 64 * 2;       // even: what follows the bitmaps in shared memory is 8-byte aligned
    const int smem_x = (BIG_STREAM_INTS + GLOBAL_BITS / 32) * (int)sizeof(int);
    constexpr int WARP_WORDS = TB_WORDS + WSTATE_INTS + Q_WORDS;     // per warp of a group kernel, beside its match hash
    constexpr int WARP_WORDS_D = TB_WORDS + WSTATE_INTS + Q_CAP;     // dense mode: one-word queue entries
    const int smem_l0 = L0_WARPS * (L0_BITS / 32 + L0_PER_WARP) * (int)sizeof(uint32_t);
    const int smem_g1 = (TSET_WORDS + G1_SLOTS + G1_BITS / 32 + G1_WARPS * (2 * G1_CAP + WARP_WORDS)) * (int)sizeof(uint32_t);
    const int smem_g2 = (TSET_WORDS + G2_SLOTS + G2_BITS / 32 + G2_WARPS * (2 * G2_CAP + WARP_WORDS)) * (int)sizeof(uint32_t);
    const int smem_gd = (TSET_WORDS + dense_words + GD_WARPS * (2 * GD_CAP + WARP_WORDS_D)) * (int)sizeof(uint32_t);
    auto* k_g1 = paper_group_kernel<G1_WARPS, G1_SLOTS, G1_BITS, G1_CAP, G1_CTAS_PER_SM, false>;
    auto* k_g2 = paper_group_kernel<G2_WARPS, G2_SLOTS, G2_BITS, G2_CAP, 1, false>;
    auto* k_gd = paper_group_kernel<GD_WARPS, 64, 32, GD_CAP, GD_CTAS_PER_SM, true>;
    if (!attr_done) {
        DCR_CUDA(cudaFuncSetAttribute(paper_edge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_x));
        DCR_CUDA(cudaFuncSetAttribute(paper_light_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_l0));
        DCR_CUDA(cudaFuncSetAttribute(k_g1, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_g1));
        DCR_CUDA(cudaFuncSetAttribute(k_g2, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_g2));
        const int smem_gd_max = (TSET_WORDS + DENSE_MAX_N / 32 + GD_WARPS * (2 * GD_CAP + WARP_WORDS_D)) * (int)sizeof(uint32_t);
        DCR_CUDA(cudaFuncSetAttribute(k_gd, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_gd_max));
        attr_done = true;
    }
    // The class kernels are independent (disjoint edges, disjoint outputs).  They are launched on streams forked
    // from `st` so that, as the persistent CTAs of one class run out of work, CTAs of another class take over the
    // freed SMs instead of waiting for the slowest CTA.
    constexpr int N_AUX = 3;
    cudaStream_t* aux = ax.aux;
    cudaEvent_t& ev_fork = ax.fork;
    cudaEvent_t* ev_join = ax.join;
    if (!ax.ready) {
        for (int q = 0; q < N_AUX; ++q) {
            DCR_CUDA(cudaStreamCreateWithFlags(&aux[q], cudaStreamNonBlocking));
            DCR_CUDA(cudaEventCreateWithFlags(&ev_join[q], cudaEventDisableTiming));
        }
        DCR_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
        ax.ready = true;
    }
    DCR_CUDA(cudaEventRecord(ev_fork, st));
    const int n_aux = a.dense ? 1 : N_AUX;
    for (int q = 0; q < n_aux; ++q) DCR_CUDA(cudaStreamWaitEvent(aux[q], ev_fork, 0));
    if (a.dense) {
#ifndef DCR_ONLY_LIGHT     // (tuning builds: time one of the two edge kernels alone)
        k_gd<<<sms * GD_CTAS_PER_SM, GD_WARPS * 32, smem_gd, st>>>(a, CL_G1, dense_words);
        DCR_LAUNCH_CHECK();
#endif
    } else {
        if (L.gslots) {
            paper_edge_kernel<<<L.g_ctas, BIG_THREADS, smem_x, aux[2]>>>(a, CL_X);
            DCR_LAUNCH_CHECK();
        }
        k_g2<<<sms, G2_WARPS * 32, smem_g2, st>>>(a, CL_G2, 0);
        DCR_LAUNCH_CHECK();
        k_g1<<<sms * G1_CTAS_PER_SM, G1_WARPS * 32, smem_g1, aux[1]>>>(a, CL_G1, 0);
        DCR_LAUNCH_CHECK();
    }
#ifndef DCR_ONLY_GROUP
    paper_light_warp_kernel<<<sms * L0_CTAS_PER_SM, L0_WARPS * 32, smem_l0, aux[0]>>>(a);
    DCR_LAUNCH_CHECK();
#endif
    for (int q = 0; q < n_aux; ++q) {
        DCR_CUDA(cudaEventRecord(ev_join[q], aux[q]));
        DCR_CUDA(cudaStreamWaitEvent(st, ev_join[q], 0));
    }
    if (value_kernel) {
        paper_value_kernel<<<tb, 256, 0, st>>>(a);
        DCR_LAUNCH_CHECK();
    }
    if (ev_edge_end) DCR_CUDA(cudaEventRecord((cudaEvent_t)ev_edge_end, st));
    return 0;
}

extern "C" int dcr_bfc_paper(const int32_t* rowptr, const int32_t* colidx, int n, int max_degree,
                             const int32_t* esrc, const int32_t* edst, int64_t e_first, int64_t e_stride,
                             int64_t count, int32_t* out_tri, int32_t* out_sq_i, int32_t* out_sq_j,
                             int32_t* out_gamma, double* out_bfc, void* scratch, int64_t scratch_bytes,
                             void* ev_edge_begin, void* ev_edge_end, void* stream) {
    return paper_pass(rowptr, colidx, n, max_degree, esrc, edst, e_first, e_stride, count, out_tri, out_sq_i, out_sq_j,
                      out_gamma, out_bfc, scratch, scratch_bytes, ev_edge_begin, ev_edge_end, stream, true);
}

#ifdef DCR_PAPER_TRACE
extern "C" int dcr_paper_trace_read(unsigned long long* host_out, int n_ctas) {
    return cudaMemcpyFromSymbol(host_out, dcr::g_trace, sizeof(unsigned long long) * 6 * n_ctas) == cudaSuccess ? 0 : 1;
}
extern "C" int dcr_paper_trace_counters(unsigned long long* host_out, int reset) {
    if (cudaMemcpyFromSymbol(host_out, dcr::g_trace_cnt, sizeof(unsigned long long) * 8) != cudaSuccess) return 1;
    if (reset) {
        unsigned long long z[8] = {0};
        if (cudaMemcpyToSymbol(dcr::g_trace_cnt, z, sizeof(z)) != cudaSuccess) return 1;
    }
    return 0;
}
#endif

// ------------------------------------------------------------------------------------------------------------
// multi-GPU: re-interleave the all-gathered per-rank shards (rank r holds edges e = r + t*world at local t)
// ------------------------------------------------------------------------------------------------------------
namespace dcr {
__global__ void unshard_kernel(const unsigned char* __restrict__ gathered, int world, int64_t chunk, int64_t n_edges,
                               int32_t* __restrict__ tri, int32_t* __restrict__ sq_i, int32_t* __restrict__ sq_j,
                               int32_t* __restrict__ gamma, double* __restrict__ bfc) {
    // per-rank block layout (bytes): bfc[chunk] f64 | tri[chunk] | sq_i[chunk] | sq_j[chunk] | gamma[chunk] i32
    const int64_t block = chunk * 24;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n_edges; e += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(e % world);
        const int64_t t = e / world;
        const unsigned char* base = gathered + r * block;
        bfc[e] = ((const double*)base)[t];
        const int32_t* ints = (const int32_t*)(base + chunk * 8);
        tri[e] = ints[t];
        sq_i[e] = ints[chunk + t];
        sq_j[e] = ints[2 * chunk + t];
        gamma[e] = ints[3 * chunk + t];
    }
}
}  // namespace dcr

extern "C" int dcr_bfc_paper_unshard(const void* gathered, int world, int64_t chunk, int64_t n_edges, int32_t* out_tri,
                                     int32_t* out_sq_i, int32_t* out_sq_j, int32_t* out_gamma, double* out_bfc,
                                     void* stream) {
    if (n_edges <= 0) return 0;
    if (world <= 0 || chunk * world < n_edges) { set_error("dcr_bfc_paper_unshard: bad shard geometry"); return 1; }
    const int ctas = (int)std::min<int64_t>((n_edges + 255) / 256, (int64_t)sm_count() * 8);
    unshard_kernel<<<ctas, 256, 0, (cudaStream_t)stream>>>((const unsigned char*)gathered, world, chunk, n_edges,
                                                          out_tri, out_sq_i, out_sq_j, out_gamma, out_bfc);
    DCR_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// multi-GPU, contiguous edge ranges: the value kernel of a rank doubles as the all-gather.  Every rank owns the
// FULL result arrays (indexed by edge id) in a buffer its peers can write (CUDA IPC over NVLink / NVSwitch); rank r
// computes the edges [e_lo, e_lo + count) and its closing kernel stores each edge's five results at the edge's own
// position in EVERY rank's buffer — no staging block, no collective call, no re-interleave pass.  Two small flag
// arrays per buffer carry the hand-shake: ready[p] = "rank p has passed the start of pass k" (its consumers of the
// previous pass are done: its buffer may be overwritten), done[p] = "all of rank p's results of pass k have landed".
// ------------------------------------------------------------------------------------------------------------
namespace dcr {

// bfc_naive.py:31-32 / :39-40 for the edges [e_lo, e_lo + count) + the fused all-gather (see above)
__global__ void __launch_bounds__(256) paper_value_exchange_kernel(PaperArgs a, CommView c) {
    __shared__ int s_last;
    unsigned char* mine = c.peers[c.rank];
    CommFlags* fl = comm_flags(mine, c.flag_off);
    if (threadIdx.x < c.world && threadIdx.x != c.rank) {           // the peers' buffers are free to take pass `epoch`
        const unsigned long long t0 = comm_now();
        while ((int)(ld_acquire_sys(&fl->ready[threadIdx.x]) - c.epoch) < 0) {
            if (comm_now() - t0 > COMM_TIMEOUT_NS) { fl->error = 1u; break; }
            __nanosleep(200);
        }
    }
    __syncthreads();
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < a.count) {
        const int64_t e = a.e_first + t;
        const int i = a.esrc[e], j = a.edst[e];
        const int di = a.rowptr[i + 1] - a.rowptr[i], dj = a.rowptr[j + 1] - a.rowptr[j];
        const int tri = a.out_tri[t], sq_i = a.out_sq_i[t], sq_j = a.out_sq_j[t], gamma = a.out_gamma[t];
        const double v = min(di, dj) <= 1 ? 0.0 : paper_value(di, dj, tri, sq_i, sq_j, gamma);   // :18-19 -> 0
        a.out_bfc[t] = v;
        for (int q = 1; q < c.world; ++q) {
            const int p = (c.rank + q) % c.world;                    // every rank starts with a different peer
            unsigned char* buf = c.peers[p];
            ((double*)buf)[e] = v;
            int32_t* ints = (int32_t*)(buf + c.chunk * 8);
            ints[e] = tri;
            ints[c.chunk + e] = sq_i;
            ints[2 * c.chunk + e] = sq_j;
            ints[3 * c.chunk + e] = gamma;
        }
    }
    if (c.world == 1) return;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(&fl->blocks_done, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {                                                    // everything this rank had to deliver is on its way
        __threadfence_system();
        if (threadIdx.x == 0) fl->blocks_done = 0u;
        if (threadIdx.x < c.world && threadIdx.x != c.rank)
            st_release_sys(&comm_flags(c.peers[threadIdx.x], c.flag_off)->done[c.rank], c.epoch);
    }
}

}  // namespace dcr

extern "C" int dcr_bfc_paper_sharded(const int32_t* rowptr, const int32_t* colidx, int n, int max_degree,
                                     const int32_t* esrc, const int32_t* edst, int64_t e_lo, int64_t count,
                                     dcr_comm* c, void* scratch, int64_t scratch_bytes, void* ev_edge_begin,
                                     void* ev_edge_end, void* stream) {
    if (!c) { set_error("dcr_bfc_paper_sharded: comm is NULL"); return 1; }
    if (!c->connected) { set_error("dcr_bfc_paper_sharded: dcr_comm_connect has not been called"); return 1; }
    if (e_lo < 0 || count < 0 || e_lo + count > c->n_edges) { set_error("dcr_bfc_paper_sharded: edge range outside [0, n_edges)"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    CommView v;
    v.peers = c->d_peers; v.rank = c->rank; v.world = c->world; v.chunk = c->chunk; v.flag_off = c->flag_off;
    v.epoch = ++c->epoch;
    if (c->world > 1) {
        comm_ready_kernel<<<1, COMM_MAX_WORLD, 0, st>>>(v);
        DCR_LAUNCH_CHECK();
    }
    double* bfc = (double*)c->local + e_lo;
    int32_t* ints = (int32_t*)(c->local + c->chunk * 8);
    int32_t *tri = ints + e_lo, *sq_i = ints + c->chunk + e_lo, *sq_j = ints + 2 * c->chunk + e_lo, *gamma = ints + 3 * c->chunk + e_lo;
    if (count > 0) {
        const int rc = paper_pass(rowptr, colidx, n, max_degree, esrc, edst, e_lo, 1, count, tri, sq_i, sq_j, gamma, bfc,
                                  scratch, scratch_bytes, ev_edge_begin, nullptr, stream, false);
        if (rc) return rc;
    }
    PaperArgs a{};
    a.rowptr = rowptr; a.colidx = colidx; a.esrc = esrc; a.edst = edst;
    a.e_first = e_lo; a.e_stride = 1; a.count = count;
    a.out_tri = tri; a.out_sq_i = sq_i; a.out_sq_j = sq_j; a.out_gamma = gamma; a.out_bfc = bfc;
    // (an empty range still takes part in the hand-shake: one block that only signals)
    const unsigned blocks = (unsigned)std::max<int64_t>(1, (count + 255) / 256);
    paper_value_exchange_kernel<<<blocks, 256, 0, st>>>(a, v);
    DCR_LAUNCH_CHECK();
    if (ev_edge_end) DCR_CUDA(cudaEventRecord((cudaEvent_t)ev_edge_end, st));
    if (c->world > 1) {
        comm_wait_kernel<<<1, COMM_MAX_WORLD, 0, st>>>(v);
        DCR_LAUNCH_CHECK();
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// work estimate per undirected edge, for cutting the edge list into contiguous ranges of equal WORK (SURVEY.md §8e):
// the entries the pass streams for the edge (the cheaper side's 2-hop lists) plus a per-head and a per-edge term.
// ------------------------------------------------------------------------------------------------------------
namespace dcr {
__global__ void edge_cost_kernel(const int32_t* __restrict__ rowptr, const int64_t* __restrict__ node_s,
                                 const int32_t* __restrict__ esrc, const int32_t* __restrict__ edst, int64_t n_edges,
                                 int64_t* __restrict__ cost) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_edges) return;
    const int i = esrc[e], j = edst[e];
    const int64_t di = rowptr[i + 1] - rowptr[i], dj = rowptr[j + 1] - rowptr[j];
    if (min(di, dj) <= 1) { cost[e] = 2; return; }
    const int64_t ca = node_s[j] - di, cb = node_s[i] - dj;
    const bool swapped = cb < ca;                    // stream i's side
    const int64_t stream = swapped ? cb : ca, heads = swapped ? di : dj, da = swapped ? dj : di;
    // Relative cost per streamed entry of the three paths, fitted (non-negative least squares, profiles/cost_model_fit.py)
    // to the measured edge-kernel times of 44 contiguous ranges of the arxiv-shaped edge list: the d_a <= 128 warp path
    // 0.5 (its kernel runs in the shadow of the group kernel), the group kernel's warp path 2.3 x (1 + d_a / 1400) — a
    // hub's streams carry more true neighbours of the tested endpoint: more candidates per element —, one CTA per edge 2.3.
    const int64_t w8 = stream > COOP_G ? 18 : (da > CLASS_DA0 ? 18 + da / 90 : 4);      // weights x 8
    cost[e] = (w8 * stream) / 8 + 24 * heads + 160;
}
}  // namespace dcr

extern "C" int dcr_bfc_paper_edge_cost(const int32_t* rowptr, const int32_t* colidx, int n, const int32_t* esrc,
                                       const int32_t* edst, int64_t n_edges, int64_t* out_cost, int64_t* node_s_scratch,
                                       void* stream) {
    if (n <= 0 || n_edges <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    node_s_kernel<<<(unsigned)((n + 31) / 32), 256, 0, st>>>(rowptr, colidx, n, node_s_scratch);
    DCR_LAUNCH_CHECK();
    edge_cost_kernel<<<(unsigned)((n_edges + 255) / 256), 256, 0, st>>>(rowptr, node_s_scratch, esrc, edst, n_edges, out_cost);
    DCR_LAUNCH_CHECK();
    return 0;
}
