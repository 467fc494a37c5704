// Technology mapping of AIGs onto single MIG / XMG / XAG gates: 3-input cut enumeration with truth tables, area-flow
// ranking, and the cover (deepgate/mapping.py, include/mgv_b200.h "mapping").
//
// One thread per AND node, one launch per level that holds AND nodes, in level order: a node reads only the cut sets of
// nodes at lower levels, written by earlier launches, so no grid barrier is needed.  A node's cuts are built by its one
// thread in a fixed order from its fan-ins' kept cuts, and every quantity is an integer, so the result does not depend on
// the batch, the launch shape or the run.  tests/map_oracle.py is the per-node Python reference of the same definitions.
//
// Cut: up to 3 distinct non-NOT leaves in ascending id; 8-bit truth table with leaf i as variable i, replicated over the
// unused variables.  Merge of an AND node v: fan-ins resolved through NOT chains to literals (u0, c0) <= (u1, c1); each
// fan-in offers [base cut, its kept cuts in rank order], where the base cut is the trivial cut {u} or, for an alias u,
// u's alias cut alone; unions of at most 3 leaves in (i, j) order, table = (t_i ^ c0) & (t_j ^ c1) over the union,
// support reduced; a union is dropped when a cut with a subset of its leaves came first (so duplicates keep the first
// table), and it removes the earlier cuts whose leaves are a strict superset of its own.  Pair (0, 0) is the structural
// cut {u0, u1}, an AND2 with polarities.
// A cut of at most 1 leaf makes v an alias (a constant, or a literal of a leaf): the best-ranked such cut is v's only cut.
// Otherwise the candidates are ranked by (flow, leaves, leaf ids), flow = cost + sum(flow(leaf) / fanout(leaf)) in
// saturating uint32, cost = MAP_UNIT for a cut whose table matches a single gate and 2 MAP_UNIT otherwise; the first
// MAP_C are kept, the structural cut in the last slot if it ranks lower.  v's best cut is its best-ranked matched cut,
// and flow(v) its flow.
#include "mgv_common.cuh"

namespace {

constexpr int MAP_C = 16;                                  // kept cuts per node
constexpr int MAP_CAND = (MAP_C + 1) * (MAP_C + 1);        // unions of two fan-ins' [base, kept cuts]
constexpr uint32_t MAP_UNIT = 256;                         // area-flow cost of one gate
constexpr int CODE_AND = 1, CODE_NOT = 2;                  // AIG codes (dg_ae_model_aig.py)
constexpr int32_t NO_ALIAS = -3;
constexpr int THREADS = 128;

struct Cut {
    int32_t l[3];
    uint32_t kt;                                           // table | leaves << 8
};

__device__ __forceinline__ int cut_k(const Cut& c) { return (int)(c.kt >> 8); }
__device__ __forceinline__ uint32_t cut_tt(const Cut& c) { return c.kt & 0xFFu; }

__device__ __forceinline__ Cut load_cut(const int4* p) {
    const int4 q = *p;
    Cut c;
    c.l[0] = q.x; c.l[1] = q.y; c.l[2] = q.z; c.kt = (uint32_t)q.w;
    return c;
}

__device__ __forceinline__ void store_cut(int4* p, const Cut& c) { *p = make_int4(c.l[0], c.l[1], c.l[2], (int)c.kt); }

// Literal 2 u + c of the non-NOT node at the end of v's NOT chain.
__device__ __forceinline__ int resolve(const int32_t* __restrict__ code, const int32_t* __restrict__ in_ptr,
                                       const int32_t* __restrict__ in_src, int v) {
    int c = 0;
    while (code[v] == CODE_NOT) {
        v = in_src[in_ptr[v]];
        c ^= 1;
    }
    return 2 * v + c;
}

// Table `tt` over `leaves` (k of them) re-expressed over the sorted union `u` (ku leaves); leaves of the cut are in u.
__device__ __forceinline__ uint32_t expand(uint32_t tt, const int32_t* leaves, int k, const int32_t* u, int ku) {
    int pos[3] = {0, 0, 0};
    for (int i = 0; i < k; ++i)
        for (int j = 0; j < ku; ++j)
            if (u[j] == leaves[i]) pos[i] = j;
    uint32_t out = 0;
    for (int m = 0; m < 8; ++m) {
        int idx = 0;
        for (int i = 0; i < k; ++i) idx |= ((m >> pos[i]) & 1) << i;
        out |= ((tt >> idx) & 1u) << m;
    }
    return out;
}

// Drops the leaves the table does not depend on (in place).
__device__ __forceinline__ void reduce_support(Cut& c) {
    const uint32_t neg[3] = {0x55u, 0x33u, 0x0Fu};
    const uint32_t tt = cut_tt(c);
    const int k = cut_k(c);
    int keep[3], nk = 0;
    for (int i = 0; i < k; ++i)
        if (((tt >> (1 << i)) ^ tt) & neg[i]) keep[nk++] = i;
    if (nk == k) return;
    uint32_t out = 0;
    for (int m = 0; m < 8; ++m) {
        int idx = 0;
        for (int j = 0; j < nk; ++j) idx |= ((m >> j) & 1) << keep[j];
        out |= ((tt >> idx) & 1u) << m;
    }
    Cut r;
    r.l[0] = r.l[1] = r.l[2] = -1;
    for (int j = 0; j < nk; ++j) r.l[j] = c.l[keep[j]];
    r.kt = out | ((uint32_t)nk << 8);
    c = r;
}

// Leaves of a are a subset of those of b (both ascending).
__device__ __forceinline__ bool subset(const Cut& a, const Cut& b) {
    const int ka = cut_k(a), kb = cut_k(b);
    if (ka > kb) return false;
    int j = 0;
    for (int i = 0; i < ka; ++i) {
        while (j < kb && b.l[j] < a.l[i]) ++j;
        if (j == kb || b.l[j] != a.l[i]) return false;
        ++j;
    }
    return true;
}

// Rank order: flow, then fewer leaves, then leaf ids.
__device__ __forceinline__ bool before(uint32_t fa, const Cut& a, uint32_t fb, const Cut& b) {
    if (fa != fb) return fa < fb;
    if (cut_k(a) != cut_k(b)) return cut_k(a) < cut_k(b);
    for (int i = 0; i < cut_k(a); ++i)
        if (a.l[i] != b.l[i]) return a.l[i] < b.l[i];
    return false;
}

struct MapArgs {
    const int32_t* code;
    const int32_t* in_ptr;
    const int32_t* in_src;
    const int32_t* order;
    const int32_t* match;                                  // [256] per table: gate | mask << 3 | out << 6, or -1
    const int32_t* fanout;
    int4* cuts;                                            // [N][MAP_C]
    int32_t* ncut;
    int4* best;                                            // [N]: leaves, table | leaves << 8
    int32_t* best_match;
    uint32_t* flow;
    int32_t* alias;
    int32_t N;
};

__global__ void __launch_bounds__(256) map_init_kernel(const MapArgs a, int32_t* fanout) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= a.N) return;
    a.ncut[v] = 0;
    a.best[v] = make_int4(-1, -1, -1, 0);
    a.best_match[v] = -1;
    a.flow[v] = 0;
    a.alias[v] = NO_ALIAS;
    if (a.code[v] != CODE_AND) return;
    for (int q = a.in_ptr[v]; q < a.in_ptr[v + 1]; ++q)
        atomicAdd(fanout + (resolve(a.code, a.in_ptr, a.in_src, a.in_src[q]) >> 1), 1);
}

// Fan-in u's offered cut i: i = 0 the base cut, i >= 1 its kept cut i - 1.
__device__ __forceinline__ Cut offered(const MapArgs& a, int u, int i) {
    if (i == 0 && a.alias[u] == NO_ALIAS) {
        Cut c;
        c.l[0] = u; c.l[1] = c.l[2] = -1;
        c.kt = 0xAAu | (1u << 8);
        return c;
    }
    return load_cut(a.cuts + (size_t)u * MAP_C + (a.alias[u] == NO_ALIAS ? i - 1 : 0));
}

__device__ __forceinline__ uint32_t cut_flow(const MapArgs& a, const Cut& c) {
    uint64_t f = a.match[cut_tt(c)] >= 0 ? MAP_UNIT : 2 * MAP_UNIT;
    for (int i = 0; i < cut_k(c); ++i) {
        const int u = c.l[i];
        const int fo = a.fanout[u] > 1 ? a.fanout[u] : 1;
        f += a.flow[u] / (uint32_t)fo;
    }
    return f > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)f;
}

__global__ void __launch_bounds__(THREADS, 1) map_cuts_kernel(const MapArgs a, int beg, int count) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const int v = a.order[beg + t];
    const int p = a.in_ptr[v];
    int f0 = resolve(a.code, a.in_ptr, a.in_src, a.in_src[p]);
    int f1 = resolve(a.code, a.in_ptr, a.in_src, a.in_src[p + 1]);
    if (f1 < f0) { const int s = f0; f0 = f1; f1 = s; }
    const int u0 = f0 >> 1, u1 = f1 >> 1;
    const uint32_t c0 = (f0 & 1) ? 0xFFu : 0u, c1 = (f1 & 1) ? 0xFFu : 0u;
    const int n0 = a.alias[u0] == NO_ALIAS ? 1 + a.ncut[u0] : 1;
    const int n1 = a.alias[u1] == NO_ALIAS ? 1 + a.ncut[u1] : 1;

    Cut cand[MAP_CAND];
    int n = 0;
    for (int i = 0; i < n0; ++i) {
        const Cut x = offered(a, u0, i);
        for (int j = 0; j < n1; ++j) {
            const Cut y = offered(a, u1, j);
            Cut w;                                          // sorted union of the leaves
            int kw = 0, ix = 0, iy = 0;
            const int kx = cut_k(x), ky = cut_k(y);
            bool fits = true;
            while (ix < kx || iy < ky) {
                int next;
                if (iy == ky || (ix < kx && x.l[ix] < y.l[iy])) next = x.l[ix++];
                else if (ix == kx || y.l[iy] < x.l[ix]) next = y.l[iy++];
                else { next = x.l[ix++]; ++iy; }
                if (kw == 3) { fits = false; break; }
                w.l[kw++] = next;
            }
            if (!fits) continue;
            for (int q = kw; q < 3; ++q) w.l[q] = -1;
            const uint32_t tt = ((expand(cut_tt(x), x.l, kx, w.l, kw) ^ c0) & (expand(cut_tt(y), y.l, ky, w.l, kw) ^ c1)) & 0xFFu;
            w.kt = tt | ((uint32_t)kw << 8);
            reduce_support(w);
            bool dominated = false;
            for (int q = 0; q < n && !dominated; ++q) dominated = subset(cand[q], w);
            if (dominated) continue;
            int m = 0;
            for (int q = 0; q < n; ++q)
                if (!subset(w, cand[q])) cand[m++] = cand[q];
            n = m;
            cand[n++] = w;
        }
    }

    int4* mine = a.cuts + (size_t)v * MAP_C;
    // alias: the best-ranked cut of at most one leaf
    int al = -1;
    uint32_t alf = 0;
    for (int q = 0; q < n; ++q) {
        if (cut_k(cand[q]) > 1) continue;
        const uint32_t f = cut_flow(a, cand[q]);
        if (al < 0 || before(f, cand[q], alf, cand[al])) { al = q; alf = f; }
    }
    if (al >= 0) {
        const Cut& c = cand[al];
        store_cut(mine, c);
        a.ncut[v] = 1;
        a.best[v] = make_int4(c.l[0], c.l[1], c.l[2], (int)c.kt);
        a.alias[v] = cut_k(c) == 0 ? (cut_tt(c) ? -1 : -2) : 2 * c.l[0] + (cut_tt(c) == 0x55u ? 1 : 0);
        return;
    }

    // ranking: the first MAP_C by insertion, the best matched cut, the structural cut (the first generated)
    int top[MAP_C];
    uint32_t topf[MAP_C];
    int nt = 0, bm = -1;
    uint32_t bmf = 0;
    bool structural_kept = false;
    for (int q = 0; q < n; ++q) {
        const uint32_t f = cut_flow(a, cand[q]);
        if (a.match[cut_tt(cand[q])] >= 0 && (bm < 0 || before(f, cand[q], bmf, cand[bm]))) { bm = q; bmf = f; }
        if (nt == MAP_C && !before(f, cand[q], topf[MAP_C - 1], cand[top[MAP_C - 1]])) continue;
        int s = nt < MAP_C ? nt++ : MAP_C - 1;
        while (s > 0 && before(f, cand[q], topf[s - 1], cand[top[s - 1]])) {
            top[s] = top[s - 1];
            topf[s] = topf[s - 1];
            --s;
        }
        top[s] = q;
        topf[s] = f;
    }
    for (int s = 0; s < nt; ++s) structural_kept |= top[s] == 0;
    if (!structural_kept) top[nt - 1] = 0;
    for (int s = 0; s < nt; ++s) store_cut(mine + s, cand[top[s]]);
    a.ncut[v] = nt;
    const Cut& b = cand[bm];
    a.best[v] = make_int4(b.l[0], b.l[1], b.l[2], (int)b.kt);
    a.best_match[v] = a.match[cut_tt(b)];
    a.flow[v] = bmf;
}

__global__ void __launch_bounds__(256) map_roots_kernel(const int32_t* __restrict__ code, const int32_t* __restrict__ in_ptr,
                                                        const int32_t* __restrict__ in_src, const int32_t* __restrict__ alias,
                                                        const int32_t* __restrict__ roots, int64_t n_roots,
                                                        uint8_t* __restrict__ required) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_roots) return;
    int u = resolve(code, in_ptr, in_src, roots[i]) >> 1;
    if (alias[u] != NO_ALIAS) {
        if (alias[u] < 0) return;                          // a constant
        u = alias[u] >> 1;
    }
    required[u] = 1;
}

__global__ void __launch_bounds__(256) map_cover_kernel(const int32_t* __restrict__ order, int beg, int count,
                                                        const int4* __restrict__ best, const int32_t* __restrict__ alias,
                                                        uint8_t* required) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const int v = order[beg + t];
    if (!required[v] || alias[v] != NO_ALIAS) return;
    const int4 b = best[v];
    const int k = (b.w >> 8) & 3;
    if (k > 0) required[b.x] = 1;
    if (k > 1) required[b.y] = 1;
    if (k > 2) required[b.z] = 1;
}

struct MapBufs {
    int4* cuts;
    int32_t *ncut, *fanout;
};

size_t map_layout(int64_t N, void* ws, MapBufs& b) {
    MgvArena ar(ws, ~(size_t)0);
    b.cuts = ar.take<int4>((size_t)N * MAP_C);
    b.ncut = ar.take<int32_t>(N);
    b.fanout = ar.take<int32_t>(N);
    return ar.off;
}

int check_levels(const int32_t* levels_host, int32_t n_levels, int32_t N, const char* what) {
    MGV_REQUIRE(n_levels >= 0 && (n_levels == 0 || levels_host), "%s: NULL levels_host or n_levels = %d", what, n_levels);
    for (int i = 0; i < n_levels; ++i) {
        const int beg = levels_host[2 * i], cnt = levels_host[2 * i + 1];
        MGV_REQUIRE(beg >= 0 && cnt >= 0 && (int64_t)beg + cnt <= N, "%s: level %d: segment [%d, %d + %d) outside the order "
                    "of %d nodes", what, i, beg, beg, cnt, N);
    }
    return MGV_OK;
}

}  // namespace

extern "C" size_t mgv_map_cuts_bytes(int64_t N) {
    if (N <= 0 || N > INT32_MAX) return 0;
    MapBufs b;
    return map_layout(N, nullptr, b);
}

extern "C" int mgv_map_cuts(const mgv_schedule* sch, const int32_t* code, const int32_t* match,
                            const int32_t* levels_host, int32_t n_levels, int32_t* best, int32_t* best_match,
                            uint32_t* flow, int32_t* alias, void* ws, size_t ws_bytes, mgv_stream_t stream) {
    MGV_REQUIRE(sch && code && match, "map_cuts: NULL schedule, code or match table");
    MGV_REQUIRE(best && best_match && flow && alias, "map_cuts: NULL best, best_match, flow or alias");
    const int32_t N = sch->N;
    if (N == 0) return MGV_OK;
    int rc = check_levels(levels_host, n_levels, N, "map_cuts");
    if (rc != MGV_OK) return rc;
    const size_t need = mgv_map_cuts_bytes(N);
    MGV_REQUIRE(ws && ws_bytes >= need, "map_cuts: workspace of %zu bytes, need mgv_map_cuts_bytes = %zu", ws_bytes, need);
    MapBufs b;
    map_layout(N, ws, b);
    cudaStream_t st = (cudaStream_t)stream;
    MapArgs a{code, sch->in_ptr, sch->in_src, sch->order, match, b.fanout, b.cuts, b.ncut,
              reinterpret_cast<int4*>(best), best_match, flow, alias, N};
    MGV_CUDA(cudaMemsetAsync(b.fanout, 0, (size_t)N * sizeof(int32_t), st));
    map_init_kernel<<<(N + 255) / 256, 256, 0, st>>>(a, b.fanout);
    MGV_CUDA(cudaGetLastError());
    for (int i = 0; i < n_levels; ++i) {
        const int beg = levels_host[2 * i], cnt = levels_host[2 * i + 1];
        if (cnt == 0) continue;
        map_cuts_kernel<<<(cnt + THREADS - 1) / THREADS, THREADS, 0, st>>>(a, beg, cnt);
        MGV_CUDA(cudaGetLastError());
    }
    mgv_count_launches(1 + n_levels);
    return MGV_OK;
}

extern "C" int mgv_map_cover(const mgv_schedule* sch, const int32_t* code, const int32_t* roots, int64_t n_roots,
                             const int32_t* levels_host, int32_t n_levels, const int32_t* best, const int32_t* alias,
                             uint8_t* required, mgv_stream_t stream) {
    MGV_REQUIRE(sch && code && best && alias && required, "map_cover: NULL schedule, code, best, alias or required");
    MGV_REQUIRE(n_roots >= 0 && (n_roots == 0 || roots), "map_cover: NULL roots or n_roots = %lld", (long long)n_roots);
    const int32_t N = sch->N;
    if (N == 0) return MGV_OK;
    int rc = check_levels(levels_host, n_levels, N, "map_cover");
    if (rc != MGV_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    MGV_CUDA(cudaMemsetAsync(required, 0, (size_t)N, st));
    int launches = 0;
    if (n_roots > 0) {
        map_roots_kernel<<<(unsigned)((n_roots + 255) / 256), 256, 0, st>>>(code, sch->in_ptr, sch->in_src, alias, roots,
                                                                          n_roots, required);
        MGV_CUDA(cudaGetLastError());
        ++launches;
    }
    for (int i = n_levels - 1; i >= 0; --i) {
        const int beg = levels_host[2 * i], cnt = levels_host[2 * i + 1];
        if (cnt == 0) continue;
        map_cover_kernel<<<(cnt + 255) / 256, 256, 0, st>>>(sch->order, beg, cnt, reinterpret_cast<const int4*>(best), alias,
                                                           required);
        MGV_CUDA(cudaGetLastError());
        ++launches;
    }
    mgv_count_launches(launches);
    return MGV_OK;
}
