// Bit-parallel logic simulation of a circuit batch: signal probabilities and truth-table distances (the `prob` and
// `tt_sim` labels the model trains on), 64 input patterns per machine word.
//
// Layout: sim[N][ld] uint64, ld = W rounded up to SIM_S words, so every node's slice of SIM_S words is one 32-byte sector.
// CTA b owns words [b*SIM_S, b*SIM_S + SIM_S) of every node and walks all levels of the schedule on that slice alone, with
// __syncthreads() between levels: the slices are independent, so there is no grid barrier, no cooperative launch and no
// wait that could hang.  One thread per node of the current level: load SIM_S words of each predecessor (one sector each),
// apply the gate function, store SIM_S words, and add the node's ones to ones[v] (integer atomics).
// Predecessor words are written earlier in the same kernel, so they are read with plain loads (never the non-coherent path).
//
// Sequential simulation (seq_sim_kernel): each of the 64 bits of a word is one trace of the circuit from its reset state.
// CTA b runs every clock cycle of the traces of its slice in one launch: per cycle the level walk above (primary INPUTs
// take the word of index t * T + trace word, latch INPUTs copy their state row), then every latch's next-state word is
// staged into its state row and read back by the next cycle's walk, with a __syncthreads() between -- so latch-to-latch
// chains and self-loops read the old state.  Each counted cycle adds one 64-bit atomic per node and per pair per slice,
// as logic_sim_kernel does: measured faster than 32-bit counters per (slice, node) reduced after the pass (DESIGN.md §4.7).
#include "mgv_common.cuh"

namespace {

constexpr int SIM_S = 4;            // words per CTA slice (one 32-byte sector)
constexpr int SIM_THREADS = 1024;

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {     // splitmix64 finaliser
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

struct SimArgs {
    const int32_t* order;
    const int32_t* seg_ptr;
    const int32_t* in_ptr;
    const int32_t* in_src;
    const int32_t* code;
    const int32_t* rank;
    int32_t L, streams;
    int32_t W, ld;
    int32_t mode;
    uint32_t fn_bits;               // 4 bits per code: the MGV_FN_* of code c at bits 4c .. 4c + 3
    uint64_t seed_mixed;            // mix64(seed), random mode
    int64_t first_word;
    uint64_t* sim;
    unsigned long long* ones;
};

// Word `gw` of the INPUT with circuit-local rank `r`.
__device__ __forceinline__ uint64_t input_word(const SimArgs& a, int r, int64_t gw) {
    if (a.mode == MGV_SIM_RANDOM) return mix64(a.seed_mixed ^ (((uint64_t)r << 40) | (uint64_t)gw));
    // exhaustive: pattern t = 64 gw + bit; the INPUT takes bit r of t
    if (r < 6) {                    // 0xAAAA.., 0xCCCC.., 0xF0F0.., .., 0xFFFFFFFF00000000
        const int h = 1 << r;
        return (~0ull / ((1ull << h) + 1ull)) << h;
    }
    return ((gw >> (r - 6)) & 1) ? ~0ull : 0ull;
}

__device__ __forceinline__ void load4(const uint64_t* p, uint64_t (&v)[SIM_S]) {
    const ulonglong2 lo = reinterpret_cast<const ulonglong2*>(p)[0];
    const ulonglong2 hi = reinterpret_cast<const ulonglong2*>(p)[1];
    v[0] = lo.x; v[1] = lo.y; v[2] = hi.x; v[3] = hi.y;
}

// Words [w0, w0 + SIM_S) of gate v with function fn (not INPUT, not NONE) from its predecessors' words: the one copy of
// the gate semantics, shared by logic_sim_kernel and seq_sim_kernel.
__device__ __forceinline__ void gate_words(const SimArgs& a, int v, int fn, int w0, uint64_t (&out)[SIM_S]) {
    const int p0 = a.in_ptr[v], p1 = a.in_ptr[v + 1];
    load4(a.sim + (size_t)a.in_src[p0] * a.ld + w0, out);
    if (fn == MGV_FN_NOT) {
#pragma unroll
        for (int k = 0; k < SIM_S; ++k) out[k] = ~out[k];
    } else if (fn == MGV_FN_MAJ) {
        uint64_t b[SIM_S], d[SIM_S];
        load4(a.sim + (size_t)a.in_src[p0 + 1] * a.ld + w0, b);
        load4(a.sim + (size_t)a.in_src[p0 + 2] * a.ld + w0, d);
#pragma unroll
        for (int k = 0; k < SIM_S; ++k) out[k] = (out[k] & b[k]) | (out[k] & d[k]) | (b[k] & d[k]);
    } else {
        for (int q = p0 + 1; q < p1; ++q) {
            uint64_t b[SIM_S];
            load4(a.sim + (size_t)a.in_src[q] * a.ld + w0, b);
#pragma unroll
            for (int k = 0; k < SIM_S; ++k)
                out[k] = fn == MGV_FN_AND ? (out[k] & b[k]) : fn == MGV_FN_OR ? (out[k] | b[k]) : (out[k] ^ b[k]);
        }
    }
}

__device__ __forceinline__ void store4(uint64_t* p, const uint64_t (&v)[SIM_S]) {
    reinterpret_cast<ulonglong2*>(p)[0] = make_ulonglong2(v[0], v[1]);
    reinterpret_cast<ulonglong2*>(p)[1] = make_ulonglong2(v[2], v[3]);
}

__device__ __forceinline__ int node_fn(const SimArgs& a, int c) {
    return (c >= 0 && c < MGV_NCODE) ? (int)((a.fn_bits >> (4 * c)) & 15u) : MGV_FN_NONE;
}

__global__ void __launch_bounds__(SIM_THREADS) logic_sim_kernel(const SimArgs a) {
    const int w0 = blockIdx.x * SIM_S;
    const int nw = min(SIM_S, a.W - w0);            // valid words of this slice (the last CTA may hold a partial one)
    for (int l = 0; l < a.L; ++l) {
        for (int s = 0; s < a.streams; ++s) {
            const int seg = (s * a.L + l) * MGV_NCODE;
            const int beg = a.seg_ptr[seg], end = a.seg_ptr[seg + MGV_NCODE];
            for (int t = beg + threadIdx.x; t < end; t += blockDim.x) {
                const int v = a.order[t];
                const int fn = node_fn(a, a.code[v]);       // validated before any pass
                uint64_t out[SIM_S] = {0, 0, 0, 0};
                if (fn == MGV_FN_INPUT) {
                    const int r = a.rank[v];
#pragma unroll
                    for (int k = 0; k < SIM_S; ++k) out[k] = input_word(a, r, a.first_word + w0 + k);
                } else if (fn != MGV_FN_NONE) {
                    gate_words(a, v, fn, w0, out);
                }
                store4(a.sim + (size_t)v * a.ld + w0, out);
                unsigned cnt = 0;
#pragma unroll
                for (int k = 0; k < SIM_S; ++k) cnt += k < nw ? __popcll(out[k]) : 0;
                if (cnt) atomicAdd(a.ones + v, (unsigned long long)cnt);
            }
        }
        __syncthreads();
    }
}

// One warp per pair: lanes over the pass's words, popc(a ^ b), one add per pair per pass.
__global__ void __launch_bounds__(256) pair_diff_kernel(const uint64_t* __restrict__ sim, int W, int ld,
                                                        const int64_t* __restrict__ pairs, int64_t P,
                                                        unsigned long long* __restrict__ diff) {
    const int lane = threadIdx.x & 31;
    const int64_t p = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (p >= P) return;
    const uint64_t* ra = sim + (size_t)pairs[p] * ld;
    const uint64_t* rb = sim + (size_t)pairs[P + p] * ld;
    unsigned long long cnt = 0;
    for (int w = lane; w < W; w += 32) cnt += __popcll(ra[w] ^ rb[w]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) diff[p] += cnt;
}

enum : uint32_t {
    BAD_CODE = 1, BAD_INPUT_FANIN, BAD_NO_FANIN, BAD_NOT_FANIN, BAD_MAJ_FANIN, BAD_REDUCE_FANIN, BAD_LEVEL_ORDER
};

// first[0] = min over bad nodes of (node << 8 | reason), first[1] = min bad pair index (both start at ~0).
__global__ void logic_sim_validate_kernel(const int32_t* __restrict__ in_ptr, const int32_t* __restrict__ in_src,
                                          const int32_t* __restrict__ code, const int32_t* __restrict__ level, int N,
                                          const SimArgs a, const int64_t* __restrict__ pairs, int64_t P,
                                          unsigned long long* __restrict__ first) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) {
        const int v = (int)i, c = code[v];
        const int fn = (c >= 0 && c < MGV_NCODE) ? (int)((a.fn_bits >> (4 * c)) & 15u) : MGV_FN_NONE;
        const int p0 = in_ptr[v], deg = in_ptr[v + 1] - p0;
        uint32_t why = 0;
        if (fn == MGV_FN_NONE) why = BAD_CODE;
        else if (fn == MGV_FN_INPUT) why = deg != 0 ? BAD_INPUT_FANIN : 0;
        else if (deg == 0) why = BAD_NO_FANIN;
        else if (fn == MGV_FN_NOT) why = deg != 1 ? BAD_NOT_FANIN : 0;
        else if (fn == MGV_FN_MAJ) why = deg != 3 ? BAD_MAJ_FANIN : 0;
        else why = deg < 2 ? BAD_REDUCE_FANIN : 0;
        for (int q = p0; q < p0 + deg && !why; ++q)
            if (level[in_src[q]] >= level[v]) why = BAD_LEVEL_ORDER;
        if (why) atomicMin(first, ((unsigned long long)v << 8) | why);
    }
    if (i < P) {
        const int64_t u = pairs[i], w = pairs[P + i];
        if (u < 0 || u >= N || w < 0 || w >= N) atomicMin(first + 1, (unsigned long long)i);
    }
}

int fill_args(SimArgs& a, const mgv_schedule* sch, const int32_t* code, const int32_t* fn_table_host) {
    MGV_REQUIRE(sch && code && fn_table_host, "logic_sim: NULL schedule, code or function table");
    a = SimArgs{};
    a.order = sch->order; a.seg_ptr = sch->seg_ptr; a.in_ptr = sch->in_ptr; a.in_src = sch->in_src;
    a.code = code;
    a.L = sch->L; a.streams = sch->streams > 1 ? sch->streams : 1;
    for (int c = 0; c < MGV_NCODE; ++c) {
        const int f = fn_table_host[c];
        MGV_REQUIRE(f >= MGV_FN_NONE && f <= MGV_FN_MAJ, "logic_sim: function table entry %d = %d is not an MGV_FN_* value", c, f);
        a.fn_bits |= (uint32_t)f << (4 * c);
    }
    return MGV_OK;
}

const char* reason_text(uint32_t why) {
    switch (why) {
        case BAD_CODE: return "gate code not defined for this circuit kind";
        case BAD_INPUT_FANIN: return "INPUT with predecessors";
        case BAD_NO_FANIN: return "gate with fan-in 0";
        case BAD_NOT_FANIN: return "NOT needs fan-in 1";
        case BAD_MAJ_FANIN: return "MAJ needs fan-in 3";
        case BAD_REDUCE_FANIN: return "AND / OR / XOR need fan-in >= 2";
        default: return "predecessor not at a lower level";
    }
}


// ------------------------------------------------------------------ sequential simulation
struct SeqArgs {
    SimArgs s;                      // s.W, s.first_word: the pass's trace words
    unsigned long long* diff;
    const int64_t* latches;         // [n_latch][3]: INPUT node, next-state literal, reset
    const int32_t* slot;            // [N]: latch index of a latch INPUT, -1 elsewhere
    uint64_t* state;                // [n_latch][ld]
    const int64_t* pairs;           // [2][P]
    int32_t n_latch, cycles, warmup;
    int64_t P, T;
};

__global__ void __launch_bounds__(SIM_THREADS) seq_sim_kernel(const SeqArgs q) {
    const SimArgs& a = q.s;
    const int w0 = blockIdx.x * SIM_S;
    const int nw = min(SIM_S, a.W - w0);
    for (int i = threadIdx.x; i < q.n_latch; i += blockDim.x) {           // s_0: the reset state
        const int64_t r = q.latches[3 * i + 2];
        uint64_t out[SIM_S];
        const uint64_t rank = (uint64_t)a.rank[q.latches[3 * i]];
#pragma unroll
        for (int k = 0; k < SIM_S; ++k)
            out[k] = r == 2 ? mix64(a.seed_mixed ^ ((rank << 40) | (uint64_t)(a.first_word + w0 + k))) : r ? ~0ull : 0ull;
        store4(q.state + (size_t)i * a.ld + w0, out);
    }
    __syncthreads();
    for (int t = 0; t < q.cycles; ++t) {
        const bool counted = t >= q.warmup;
        const int64_t gw = (int64_t)t * q.T + a.first_word + w0;
        for (int l = 0; l < a.L; ++l) {
            for (int s = 0; s < a.streams; ++s) {
                const int seg = (s * a.L + l) * MGV_NCODE;
                const int beg = a.seg_ptr[seg], end = a.seg_ptr[seg + MGV_NCODE];
                for (int p = beg + threadIdx.x; p < end; p += blockDim.x) {
                    const int v = a.order[p];
                    const int fn = node_fn(a, a.code[v]);
                    uint64_t out[SIM_S] = {0, 0, 0, 0};
                    if (fn == MGV_FN_INPUT) {
                        const int j = q.slot[v];
                        if (j >= 0) {
                            load4(q.state + (size_t)j * a.ld + w0, out);
                        } else {
                            const uint64_t r = (uint64_t)a.rank[v];
#pragma unroll
                            for (int k = 0; k < SIM_S; ++k) out[k] = mix64(a.seed_mixed ^ ((r << 40) | (uint64_t)(gw + k)));
                        }
                    } else if (fn != MGV_FN_NONE) {
                        gate_words(a, v, fn, w0, out);
                    }
                    store4(a.sim + (size_t)v * a.ld + w0, out);
                    if (counted) {
                        unsigned c = 0;
#pragma unroll
                        for (int k = 0; k < SIM_S; ++k) c += k < nw ? __popcll(out[k]) : 0;
                        if (c) atomicAdd(a.ones + v, (unsigned long long)c);
                    }
                }
            }
            __syncthreads();
        }
        if (counted) {
            for (int64_t p = threadIdx.x; p < q.P; p += blockDim.x) {
                uint64_t u[SIM_S], w[SIM_S];
                load4(a.sim + (size_t)q.pairs[p] * a.ld + w0, u);
                load4(a.sim + (size_t)q.pairs[q.P + p] * a.ld + w0, w);
                unsigned c = 0;
#pragma unroll
                for (int k = 0; k < SIM_S; ++k) c += k < nw ? __popcll(u[k] ^ w[k]) : 0;
                if (c) atomicAdd(q.diff + p, (unsigned long long)c);
            }
        }
        for (int i = threadIdx.x; i < q.n_latch; i += blockDim.x) {       // s_{t+1}, staged: the walk reads it next cycle
            const int64_t lit = q.latches[3 * i + 1];
            uint64_t out[SIM_S];
            if (lit < 0) {
#pragma unroll
                for (int k = 0; k < SIM_S; ++k) out[k] = lit == -1 ? ~0ull : 0ull;
            } else {
                load4(a.sim + (size_t)(lit >> 1) * a.ld + w0, out);
#pragma unroll
                for (int k = 0; k < SIM_S; ++k) out[k] ^= (lit & 1) ? ~0ull : 0ull;
            }
            store4(q.state + (size_t)i * a.ld + w0, out);
        }
        __syncthreads();
    }
}

// slot[v] = the smallest latch index whose node is v (slot starts at ~0); nodes outside [0, N) are skipped.
__global__ void latch_slot_kernel(const int64_t* __restrict__ latches, int n_latch, int64_t N, uint32_t* __restrict__ slot) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_latch) return;
    const int64_t v = latches[3 * i];
    if (v >= 0 && v < N) atomicMin(slot + v, (uint32_t)i);
}

enum : uint32_t { BAD_LATCH_NODE = 1, BAD_LATCH_NOT_INPUT, BAD_LATCH_TWICE, BAD_LATCH_NEXT, BAD_LATCH_CIRCUIT, BAD_LATCH_RESET };

// first = min over bad latches of (latch << 8 | reason), starting at ~0.
__global__ void seq_sim_validate_kernel(const int64_t* __restrict__ latches, int n_latch, int64_t N,
                                        const int32_t* __restrict__ code, const int32_t* __restrict__ circuit,
                                        const uint32_t* __restrict__ slot, const SimArgs a,
                                        unsigned long long* __restrict__ first) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_latch) return;
    const int64_t v = latches[3 * i], lit = latches[3 * i + 1], r = latches[3 * i + 2];
    uint32_t why = 0;
    if (v < 0 || v >= N) why = BAD_LATCH_NODE;
    else if (node_fn(a, code[v]) != MGV_FN_INPUT) why = BAD_LATCH_NOT_INPUT;
    else if (slot[v] != (uint32_t)i) why = BAD_LATCH_TWICE;
    else if (lit < -2 || (lit >> 1) >= N) why = BAD_LATCH_NEXT;
    else if (lit >= 0 && circuit[lit >> 1] != circuit[v]) why = BAD_LATCH_CIRCUIT;
    else if (r < 0 || r > 2) why = BAD_LATCH_RESET;
    if (why) atomicMin(first, ((unsigned long long)i << 8) | why);
}

int check_cycles(int32_t cycles, int32_t warmup) {
    MGV_REQUIRE(cycles >= 1, "seq_sim: cycles = %d must be >= 1", cycles);
    MGV_REQUIRE(warmup >= 0 && warmup < cycles, "seq_sim: warmup = %d must be in [0, cycles = %d)", warmup, cycles);
    return MGV_OK;
}

size_t seq_words(int32_t W) { return (size_t)((W > 0 ? W : 0) + SIM_S - 1) / SIM_S * SIM_S; }

}  // namespace

extern "C" size_t mgv_logic_sim_bytes(int64_t N, int32_t W) {
    const size_t ld = (size_t)((W > 0 ? W : 0) + SIM_S - 1) / SIM_S * SIM_S;
    return (size_t)(N > 0 ? N : 0) * ld * sizeof(uint64_t);
}

extern "C" int mgv_logic_sim_validate(const mgv_schedule* sch, const int32_t* code, const int32_t* level,
                                      const int32_t* fn_table_host, const int64_t* pairs, int64_t P,
                                      void* ws, size_t ws_bytes, mgv_stream_t stream) {
    SimArgs a;
    int rc = fill_args(a, sch, code, fn_table_host);
    if (rc != MGV_OK) return rc;
    MGV_REQUIRE(level && ws && ws_bytes >= 2 * sizeof(unsigned long long), "logic_sim_validate: NULL level or workspace < 16 bytes");
    MGV_REQUIRE(P >= 0 && (P == 0 || pairs), "logic_sim_validate: bad pair list");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* first = (unsigned long long*)ws;
    MGV_CUDA(cudaMemsetAsync(first, 0xff, 2 * sizeof(unsigned long long), st));
    const int64_t n = sch->N > P ? (int64_t)sch->N : P;
    if (n > 0) {
        logic_sim_validate_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sch->in_ptr, sch->in_src, code, level, sch->N,
                                                                              a, pairs, P, first);
        MGV_CUDA(cudaGetLastError());
        mgv_count_launches(1);
    }
    unsigned long long host[2];
    MGV_CUDA(cudaMemcpyAsync(host, first, sizeof(host), cudaMemcpyDeviceToHost, st));
    MGV_CUDA(cudaStreamSynchronize(st));
    if (host[0] != ~0ull) {
        const int v = (int)(host[0] >> 8);
        int32_t c = 0, p[2] = {0, 0};
        MGV_CUDA(cudaMemcpy(&c, code + v, sizeof(c), cudaMemcpyDeviceToHost));
        MGV_CUDA(cudaMemcpy(p, sch->in_ptr + v, sizeof(p), cudaMemcpyDeviceToHost));
        mgv_set_error("logic_sim: node %d (code %d, fan-in %d): %s", v, c, p[1] - p[0], reason_text((uint32_t)(host[0] & 0xff)));
        return MGV_ERR_ARG;
    }
    if (host[1] != ~0ull) {
        mgv_set_error("logic_sim: pair %lld refers to a node outside [0, %d)", (long long)host[1], sch->N);
        return MGV_ERR_ARG;
    }
    return MGV_OK;
}

extern "C" int mgv_logic_sim_pass(const mgv_schedule* sch, const int32_t* code, const int32_t* input_rank,
                                  const int32_t* fn_table_host, int32_t mode, uint64_t seed, int64_t first_word, int32_t W,
                                  uint64_t* sim, uint64_t* ones, const int64_t* pairs, int64_t P, uint64_t* diff,
                                  mgv_stream_t stream) {
    SimArgs a;
    int rc = fill_args(a, sch, code, fn_table_host);
    if (rc != MGV_OK) return rc;
    MGV_REQUIRE(mode == MGV_SIM_RANDOM || mode == MGV_SIM_EXHAUSTIVE, "logic_sim_pass: mode %d", mode);
    MGV_REQUIRE(W > 0 && first_word >= 0, "logic_sim_pass: W = %d, first_word = %lld", W, (long long)first_word);
    MGV_REQUIRE(input_rank && sim && ones, "logic_sim_pass: NULL input_rank, sim or ones");
    MGV_REQUIRE(P >= 0 && (P == 0 || (pairs && diff)), "logic_sim_pass: bad pair list");
    MGV_REQUIRE(((uintptr_t)sim & 31) == 0, "logic_sim_pass: sim must be 32-byte aligned");
    if (sch->N == 0) return MGV_OK;
    a.rank = input_rank;
    a.W = W;
    a.ld = (W + SIM_S - 1) / SIM_S * SIM_S;
    a.mode = mode;
    a.seed_mixed = mix64(seed);
    a.first_word = first_word;
    a.sim = sim;
    a.ones = (unsigned long long*)ones;
    cudaStream_t st = (cudaStream_t)stream;
    logic_sim_kernel<<<(unsigned)(a.ld / SIM_S), SIM_THREADS, 0, st>>>(a);
    MGV_CUDA(cudaGetLastError());
    int launches = 1;
    if (P > 0) {
        pair_diff_kernel<<<(unsigned)((P * 32 + 255) / 256), 256, 0, st>>>(sim, W, a.ld, pairs, P, (unsigned long long*)diff);
        MGV_CUDA(cudaGetLastError());
        ++launches;
    }
    mgv_count_launches(launches);
    return MGV_OK;
}

extern "C" size_t mgv_seq_sim_bytes(int64_t N, int32_t n_latch, int32_t W) {
    const size_t n = N > 0 ? (size_t)N : 0;
    return (n + (n_latch > 0 ? (size_t)n_latch : 0)) * seq_words(W) * sizeof(uint64_t)    // sim rows, state rows
           + n * sizeof(uint32_t);                                                     // latch slot of every node
}

extern "C" int mgv_seq_sim_validate(const mgv_schedule* sch, const int32_t* code, const int32_t* fn_table_host,
                                    const int32_t* circuit, const int64_t* latches, int32_t n_latch, int32_t cycles,
                                    int32_t warmup, void* ws, size_t ws_bytes, mgv_stream_t stream) {
    SimArgs a;
    int rc = fill_args(a, sch, code, fn_table_host);
    if (rc != MGV_OK) return rc;
    rc = check_cycles(cycles, warmup);
    if (rc != MGV_OK) return rc;
    MGV_REQUIRE(n_latch >= 0 && (n_latch == 0 || (latches && circuit)), "seq_sim_validate: bad latch list");
    const size_t need = sizeof(unsigned long long) + (size_t)sch->N * sizeof(uint32_t);
    MGV_REQUIRE(ws && ws_bytes >= need, "seq_sim_validate: workspace < %zu bytes", need);
    if (n_latch == 0) return MGV_OK;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* first = (unsigned long long*)ws;
    uint32_t* slot = (uint32_t*)(first + 1);
    MGV_CUDA(cudaMemsetAsync(ws, 0xff, need, st));
    const unsigned blocks = (unsigned)((n_latch + 255) / 256);
    latch_slot_kernel<<<blocks, 256, 0, st>>>(latches, n_latch, sch->N, slot);
    MGV_CUDA(cudaGetLastError());
    seq_sim_validate_kernel<<<blocks, 256, 0, st>>>(latches, n_latch, sch->N, code, circuit, slot, a, first);
    MGV_CUDA(cudaGetLastError());
    mgv_count_launches(2);
    unsigned long long host = 0;
    MGV_CUDA(cudaMemcpyAsync(&host, first, sizeof(host), cudaMemcpyDeviceToHost, st));
    MGV_CUDA(cudaStreamSynchronize(st));
    if (host == ~0ull) return MGV_OK;
    const int i = (int)(host >> 8);
    int64_t row[3];
    MGV_CUDA(cudaMemcpy(row, latches + 3 * (size_t)i, sizeof(row), cudaMemcpyDeviceToHost));
    switch ((uint32_t)(host & 0xff)) {
        case BAD_LATCH_NODE:
            mgv_set_error("seq_sim: latch %d: node %lld is outside [0, %d)", i, (long long)row[0], sch->N);
            break;
        case BAD_LATCH_NOT_INPUT:
            mgv_set_error("seq_sim: latch %d: node %lld is not an INPUT", i, (long long)row[0]);
            break;
        case BAD_LATCH_TWICE: {
            uint32_t other = 0;
            MGV_CUDA(cudaMemcpy(&other, slot + row[0], sizeof(other), cudaMemcpyDeviceToHost));
            mgv_set_error("seq_sim: latch %d: node %lld appears twice (also latch %u)", i, (long long)row[0], other);
            break;
        }
        case BAD_LATCH_NEXT:
            mgv_set_error("seq_sim: latch %d: next-state literal %lld names a node outside [0, %d)", i, (long long)row[1],
                          sch->N);
            break;
        case BAD_LATCH_CIRCUIT:
            mgv_set_error("seq_sim: latch %d: next-state literal %lld names a node of another circuit than node %lld", i,
                          (long long)row[1], (long long)row[0]);
            break;
        default:
            mgv_set_error("seq_sim: latch %d: reset %lld is not 0, 1 or 2 (uninitialised)", i, (long long)row[2]);
    }
    return MGV_ERR_ARG;
}

extern "C" int mgv_seq_sim_pass(const mgv_schedule* sch, const int32_t* code, const int32_t* input_rank,
                                const int32_t* fn_table_host, const int64_t* latches, int32_t n_latch, uint64_t seed,
                                int64_t first_word, int32_t W, int64_t T, int32_t cycles, int32_t warmup, void* ws,
                                size_t ws_bytes, uint64_t* ones, const int64_t* pairs, int64_t P, uint64_t* diff,
                                mgv_stream_t stream) {
    SeqArgs q{};
    int rc = fill_args(q.s, sch, code, fn_table_host);
    if (rc != MGV_OK) return rc;
    rc = check_cycles(cycles, warmup);
    if (rc != MGV_OK) return rc;
    MGV_REQUIRE(W > 0 && first_word >= 0 && first_word + W <= T, "seq_sim_pass: W = %d, first_word = %lld, T = %lld", W,
                (long long)first_word, (long long)T);
    MGV_REQUIRE((double)cycles * (double)T <= (double)MGV_SEQ_MAX_WORDS, "seq_sim_pass: cycles x T = %d x %lld is above %lld "
                "input words (a word index would reach the rank bits)", cycles, (long long)T, (long long)MGV_SEQ_MAX_WORDS);
    MGV_REQUIRE(input_rank && ones, "seq_sim_pass: NULL input_rank or ones");
    MGV_REQUIRE(n_latch >= 0 && (n_latch == 0 || latches), "seq_sim_pass: bad latch list");
    MGV_REQUIRE(P >= 0 && (P == 0 || (pairs && diff)), "seq_sim_pass: bad pair list");
    const size_t need = mgv_seq_sim_bytes(sch->N, n_latch, W);
    MGV_REQUIRE(ws && ws_bytes >= need && ((uintptr_t)ws & 31) == 0, "seq_sim_pass: workspace < %zu bytes or not 32-byte aligned",
                need);
    if (sch->N == 0) return MGV_OK;
    const size_t ld = seq_words(W), N = (size_t)sch->N;
    q.s.rank = input_rank;
    q.s.W = W;
    q.s.ld = (int)ld;
    q.s.mode = MGV_SIM_RANDOM;
    q.s.seed_mixed = mix64(seed);
    q.s.first_word = first_word;
    q.s.sim = (uint64_t*)ws;
    q.s.ones = (unsigned long long*)ones;
    q.diff = (unsigned long long*)diff;
    q.latches = latches;
    q.state = q.s.sim + N * ld;
    uint32_t* slot = (uint32_t*)(q.state + (size_t)n_latch * ld);
    q.slot = (const int32_t*)slot;
    q.pairs = pairs;
    q.n_latch = n_latch; q.cycles = cycles; q.warmup = warmup;
    q.P = P; q.T = T;
    cudaStream_t st = (cudaStream_t)stream;
    MGV_CUDA(cudaMemsetAsync(slot, 0xff, N * sizeof(uint32_t), st));
    int launches = 1;
    if (n_latch > 0) {
        latch_slot_kernel<<<(unsigned)((n_latch + 255) / 256), 256, 0, st>>>(latches, n_latch, sch->N, slot);
        MGV_CUDA(cudaGetLastError());
        ++launches;
    }
    seq_sim_kernel<<<(unsigned)(ld / SIM_S), SIM_THREADS, 0, st>>>(q);
    MGV_CUDA(cudaGetLastError());
    mgv_count_launches(launches);
    return MGV_OK;
}
