// Functional equivalence classes of a circuit batch from logic-simulation words (csrc/logic_sim.cu): nodes that are equal
// on every simulated pattern, or bitwise complementary on every one, share a class.  Exhaustive mode makes this exact
// functional equivalence; random mode is equality on the simulated patterns.
//
// Signature: after each simulation pass, one warp per node reads the pass's W valid words of sim[N][ld] and adds
//   h0[v] += mix(mix(g) ^ word), h1[v] += mix(mix(g) ^ ~word)         (g = the word's global index, mod 2^64)
// and the pass holding word 0 records bit0[v] = bit 0 of it.  Sums are commutative, so they do not depend on the pass split.
// canon[v] = bit0[v] ? h1[v] : h0[v] is equal for a node and its complement.
// Grouping: key = mix(circuit ^ canon), value = node id; stable cub radix sort; in node-id order within a run, so the
// run's first value is its smallest id, the representative.  Run starts come from a head flag and a max-scan.
// Verification: every member is compared word by word with its representative, pass by pass; a mismatch, another
// circuit or a malformed assignment flags it, and the split step makes every flagged node a singleton.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "mgv_common.cuh"

namespace {

constexpr int SIM_S = 4;            // words per slice of logic_sim.cu: the row pitch ld is W rounded up to it
constexpr int WARPS = 8;            // warps per CTA of the per-node kernels

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {     // splitmix64 finaliser (as logic_sim.cu)
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__device__ __forceinline__ uint64_t warp_sum64(uint64_t s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

int ld_of(int32_t W) { return (W + SIM_S - 1) / SIM_S * SIM_S; }

unsigned warp_grid(int64_t N) { return (unsigned)((N + WARPS - 1) / WARPS); }

__global__ void __launch_bounds__(WARPS * 32) sim_signature_kernel(const uint64_t* __restrict__ sim, int64_t N, int W, int ld,
                                                                   int64_t first_word, unsigned long long* __restrict__ h0,
                                                                   unsigned long long* __restrict__ h1,
                                                                   uint8_t* __restrict__ bit0) {
    const int lane = threadIdx.x & 31;
    const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (v >= N) return;
    const uint64_t* row = sim + (size_t)v * ld;
    uint64_t s0 = 0, s1 = 0;
    for (int w = lane; w < W; w += 32) {            // words >= W of the last slice are not patterns of this pass
        const uint64_t x = __ldg(row + w), g = mix64((uint64_t)(first_word + w));
        s0 += mix64(g ^ x);
        s1 += mix64(g ^ ~x);
    }
    s0 = warp_sum64(s0);
    s1 = warp_sum64(s1);
    if (lane == 0) {
        h0[v] += s0;
        h1[v] += s1;
        if (first_word == 0) bit0[v] = (uint8_t)(__ldg(row) & 1u);
    }
}

__global__ void class_key_kernel(const unsigned long long* __restrict__ h0, const unsigned long long* __restrict__ h1,
                                 const uint8_t* __restrict__ bit0, const int32_t* __restrict__ circuit, int N,
                                 uint64_t* __restrict__ keys, int32_t* __restrict__ vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const uint64_t canon = bit0[i] ? h1[i] : h0[i];
    keys[i] = mix64((uint64_t)(uint32_t)circuit[i] ^ canon);
    vals[i] = i;
}

__global__ void class_head_kernel(const uint64_t* __restrict__ keys, int N, int32_t* __restrict__ head) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) head[i] = (i == 0 || keys[i] != keys[i - 1]) ? i : 0;
}

struct MaxOp {
    __device__ __forceinline__ int32_t operator()(int32_t a, int32_t b) const { return a > b ? a : b; }
};

__global__ void class_scatter_kernel(const int32_t* __restrict__ vals, const int32_t* __restrict__ start,
                                     const uint8_t* __restrict__ bit0, int N, int64_t* __restrict__ rep,
                                     uint8_t* __restrict__ comp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int v = vals[i], r = vals[start[i]];
    rep[v] = r;
    comp[v] = bit0[v] ^ bit0[r];
}

// One warp per node.  A representative (rep[v] == v) must have complemented 0; a member needs a representative in
// [0, N) that is its own representative, in the same circuit, with equal (complemented 0) or complementary
// (complemented 1) words.
__global__ void __launch_bounds__(WARPS * 32) class_verify_kernel(const uint64_t* __restrict__ sim, int64_t N, int W, int ld,
                                                                  const int32_t* __restrict__ circuit,
                                                                  const int64_t* __restrict__ rep,
                                                                  const uint8_t* __restrict__ comp,
                                                                  uint8_t* __restrict__ bad) {
    const int lane = threadIdx.x & 31;
    const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (v >= N) return;
    const int64_t r = rep[v];
    const uint8_t c = comp[v];
    if (r == v) {
        if (lane == 0 && c != 0) bad[v] = 1;
        return;
    }
    if (r < 0 || r >= N || rep[r] != r || circuit[r] != circuit[v] || c > 1) {
        if (lane == 0) bad[v] = 1;
        return;
    }
    const uint64_t flip = c ? ~0ull : 0ull;
    const uint64_t* a = sim + (size_t)v * ld;
    const uint64_t* b = sim + (size_t)r * ld;
    uint64_t d = 0;
    for (int w = lane; w < W; w += 32) d |= __ldg(a + w) ^ __ldg(b + w) ^ flip;
    if (__any_sync(0xffffffffu, d != 0) && lane == 0) bad[v] = 1;
}

__global__ void class_split_kernel(int64_t N, int64_t* __restrict__ rep, uint8_t* __restrict__ comp,
                                   const uint8_t* __restrict__ bad, unsigned long long* __restrict__ count) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= N || !bad[v]) return;
    rep[v] = v;
    comp[v] = 0;
    atomicAdd(count, 1ull);
}

struct GroupBufs {
    uint64_t *keys_in, *keys_out;
    int32_t *vals_in, *vals_out, *head, *start;
    void* temp;
    size_t temp_bytes;
};

// Lays the grouping buffers out over `ws` (ws may be NULL: sizing only).  Returns the bytes needed.
size_t group_layout(int64_t N, void* ws, GroupBufs& b) {
    const int n = (int)N;
    size_t sort_bytes = 0, scan_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                    (const int32_t*)nullptr, (int32_t*)nullptr, n, 0, 64);
    cub::DeviceScan::InclusiveScan(nullptr, scan_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, MaxOp(), n);
    MgvArena ar(ws, ~(size_t)0);
    b.keys_in = ar.take<uint64_t>(N);
    b.keys_out = ar.take<uint64_t>(N);
    b.vals_in = ar.take<int32_t>(N);
    b.vals_out = ar.take<int32_t>(N);
    b.head = ar.take<int32_t>(N);
    b.start = ar.take<int32_t>(N);
    b.temp_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
    b.temp = ar.take<char>(b.temp_bytes);
    return ar.off;
}

}  // namespace

extern "C" int mgv_sim_signature_pass(const uint64_t* sim, int64_t N, int32_t W, int64_t first_word, uint64_t* h0,
                                      uint64_t* h1, uint8_t* bit0, mgv_stream_t stream) {
    MGV_REQUIRE(N >= 0 && N <= INT32_MAX, "sim_signature_pass: N = %lld", (long long)N);
    MGV_REQUIRE(W > 0 && first_word >= 0, "sim_signature_pass: W = %d, first_word = %lld", W, (long long)first_word);
    if (N == 0) return MGV_OK;
    MGV_REQUIRE(sim, "sim_signature_pass: NULL sim");
    MGV_REQUIRE(h0 && h1, "sim_signature_pass: NULL h0 or h1");
    MGV_REQUIRE(bit0, "sim_signature_pass: NULL bit0");
    cudaStream_t st = (cudaStream_t)stream;
    sim_signature_kernel<<<warp_grid(N), WARPS * 32, 0, st>>>(sim, N, W, ld_of(W), first_word, (unsigned long long*)h0,
                                                             (unsigned long long*)h1, bit0);
    MGV_CUDA(cudaGetLastError());
    mgv_count_launches(1);
    return MGV_OK;
}

extern "C" size_t mgv_sim_classes_bytes(int64_t N) {
    if (N <= 0 || N > INT32_MAX) return 0;
    GroupBufs b;
    return group_layout(N, nullptr, b);
}

extern "C" int mgv_sim_classes_group(const uint64_t* h0, const uint64_t* h1, const uint8_t* bit0, const int32_t* circuit,
                                     int64_t N, int64_t* rep, uint8_t* complemented, void* ws, size_t ws_bytes,
                                     mgv_stream_t stream) {
    MGV_REQUIRE(N >= 0 && N <= INT32_MAX, "sim_classes_group: N = %lld", (long long)N);
    if (N == 0) return MGV_OK;
    MGV_REQUIRE(h0 && h1, "sim_classes_group: NULL h0 or h1");
    MGV_REQUIRE(bit0, "sim_classes_group: NULL bit0");
    MGV_REQUIRE(circuit, "sim_classes_group: NULL circuit");
    MGV_REQUIRE(rep && complemented, "sim_classes_group: NULL rep or complemented");
    const size_t need = mgv_sim_classes_bytes(N);
    MGV_REQUIRE(ws && ws_bytes >= need, "sim_classes_group: workspace of %zu bytes, need mgv_sim_classes_bytes = %zu",
                ws_bytes, need);
    GroupBufs b;
    group_layout(N, ws, b);
    const int n = (int)N, blocks = (n + 255) / 256;
    cudaStream_t st = (cudaStream_t)stream;
    class_key_kernel<<<blocks, 256, 0, st>>>((const unsigned long long*)h0, (const unsigned long long*)h1, bit0, circuit, n,
                                             b.keys_in, b.vals_in);
    MGV_CUDA(cudaGetLastError());
    size_t tb = b.temp_bytes;
    MGV_CUDA(cub::DeviceRadixSort::SortPairs(b.temp, tb, b.keys_in, b.keys_out, b.vals_in, b.vals_out, n, 0, 64, st));
    class_head_kernel<<<blocks, 256, 0, st>>>(b.keys_out, n, b.head);
    MGV_CUDA(cudaGetLastError());
    tb = b.temp_bytes;
    MGV_CUDA(cub::DeviceScan::InclusiveScan(b.temp, tb, b.head, b.start, MaxOp(), n, st));
    class_scatter_kernel<<<blocks, 256, 0, st>>>(b.vals_out, b.start, bit0, n, rep, complemented);
    MGV_CUDA(cudaGetLastError());
    mgv_count_launches(5);
    return MGV_OK;
}

extern "C" int mgv_sim_classes_verify_pass(const uint64_t* sim, int64_t N, int32_t W, const int32_t* circuit,
                                           const int64_t* rep, const uint8_t* complemented, uint8_t* bad,
                                           mgv_stream_t stream) {
    MGV_REQUIRE(N >= 0 && N <= INT32_MAX, "sim_classes_verify_pass: N = %lld", (long long)N);
    MGV_REQUIRE(W > 0, "sim_classes_verify_pass: W = %d", W);
    if (N == 0) return MGV_OK;
    MGV_REQUIRE(sim, "sim_classes_verify_pass: NULL sim");
    MGV_REQUIRE(circuit, "sim_classes_verify_pass: NULL circuit");
    MGV_REQUIRE(rep && complemented, "sim_classes_verify_pass: NULL rep or complemented");
    MGV_REQUIRE(bad, "sim_classes_verify_pass: NULL bad");
    cudaStream_t st = (cudaStream_t)stream;
    class_verify_kernel<<<warp_grid(N), WARPS * 32, 0, st>>>(sim, N, W, ld_of(W), circuit, rep, complemented, bad);
    MGV_CUDA(cudaGetLastError());
    mgv_count_launches(1);
    return MGV_OK;
}

extern "C" int mgv_sim_classes_split(int64_t N, int64_t* rep, uint8_t* complemented, const uint8_t* bad, void* ws,
                                     size_t ws_bytes, int64_t* n_split_host, mgv_stream_t stream) {
    MGV_REQUIRE(N >= 0 && N <= INT32_MAX, "sim_classes_split: N = %lld", (long long)N);
    MGV_REQUIRE(n_split_host, "sim_classes_split: NULL n_split_host");
    MGV_REQUIRE(ws && ws_bytes >= sizeof(unsigned long long), "sim_classes_split: NULL ws or ws_bytes < 8");
    *n_split_host = 0;
    if (N == 0) return MGV_OK;
    MGV_REQUIRE(rep && complemented, "sim_classes_split: NULL rep or complemented");
    MGV_REQUIRE(bad, "sim_classes_split: NULL bad");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* count = (unsigned long long*)ws;
    MGV_CUDA(cudaMemsetAsync(count, 0, sizeof(unsigned long long), st));
    class_split_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(N, rep, complemented, bad, count);
    MGV_CUDA(cudaGetLastError());
    mgv_count_launches(1);
    unsigned long long host = 0;
    MGV_CUDA(cudaMemcpyAsync(&host, count, sizeof(host), cudaMemcpyDeviceToHost, st));
    MGV_CUDA(cudaStreamSynchronize(st));
    *n_split_host = (int64_t)host;
    return MGV_OK;
}
