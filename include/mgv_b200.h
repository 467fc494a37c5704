/*
 * mgv_b200 -- C ABI of the B200 (sm_100a) level-synchronous DAG message-passing library.
 *
 * This is the drop-in boundary for the hot path of 959AI994/Multi-Gate-VAE
 * (DG_VAE/deepgate).  The reference has no native code; each entry point below
 * replaces the Python/PyG code cited next to it (paths relative to
 * /root/reference/DG_VAE/deepgate).  The host-side mirror of the reference's
 * Python API (multi-gate-vae_b200/deepgate) binds these with ctypes.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host;
 *  - the caller (PyTorch) owns every buffer; the library allocates nothing
 *    persistent and frees nothing; workspaces are caller-provided and sized by
 *    the *_workspace_bytes() helpers;
 *  - every call takes the CUDA stream explicitly and is asynchronous on it,
 *    except where "synchronises" is stated;
 *  - return value: 0 = ok, negative = error; mgv_last_error_string() gives the
 *    message (thread-local).  No CPU fallback exists anywhere in the library.
 *  - re-entrant, no global mutable state, no cudaSetDevice: the current device
 *    of the calling thread must be the one that owns the pointers.
 *
 * Vocabulary: node = gate or primary input; level = ASAP topological level
 * (top_sort); code = gate code 0..5 {INPUT, MAJ, NOT, AND, OR, XOR} (AIG: AND=1,
 * NOT=2); D = dim_hidden = 64 (compile-time constant of the kernels).
 */
#ifndef MGV_B200_H
#define MGV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MGV_D 64                 /* dim_hidden the kernels are specialised for (config.py:13)   */
#define MGV_NCODE 8              /* code buckets per level: 0..5 real codes, 6 = other, 7 unused */
#define MGV_CODE_SHIFT 28        /* out_pack = dst | (code(dst) << 28)                          */
#define MGV_MAX_FEAT 8           /* struct encoder: dim_feature <= 8 (config.py:14 default 6)   */
#define MGV_TILE_ROWS 128        /* nodes per tensor-core tile (UMMA M)                          */
#define MGV_TILE_WAVE_COST 128   /* per dependent neighbour wave (= largest degree of the tile) of the tile cost model    */
#define MGV_TILE_FIXED_COST 2048 /* per-tile fixed cost, in node-row reads, of the tile cost model */

/* Floats per gate-code weight block of the level sweep (see mgv_sweep_pack layout below). */
#define MGV_SWEEP_PACK_FLOATS 66112
/* Floats per gate-code gradient block returned by the backward sweep. */
#define MGV_SWEEP_GRAD_FLOATS 33344
/* Floats per (encoder, direction) weight block of the struct encoder. */
#define MGV_STRUCT_PACK_FLOATS 28416
#define MGV_STRUCT_GRAD_FLOATS 28416

typedef void* mgv_stream_t;      /* cudaStream_t */

const char* mgv_last_error_string(void);
int mgv_version(void);
/* Number of SMs of the current device (grid sizing for the persistent kernels). */
int mgv_sm_count(void);
/* Kernels launched by this library in this process so far (statistics only). */
long long mgv_kernel_launches(void);

/* ------------------------------------------------------------------ schedule (integer work)
 * In/out-edge CSR by node id, ascending ORIGINAL EDGE ID inside a node -- the order in which
 * utils/dag_utils.py:91-105 `subgraph` concatenates a node's incoming edges.
 *   edge_index  int64 [2,E] row-major (row 0 = src/"parent", row 1 = dst/"child")
 *   code        int32 [N] or NULL (then out_pack carries no code bits)
 *   in_ptr[N+1], in_src[E]                      : predecessors of node v = in_src[in_ptr[v] .. in_ptr[v+1])
 *   out_ptr[N+1], out_pack[E], out_slot[E]      : successors; out_slot = position of that edge in in_src
 *   err_flag    int32 device word or NULL.  NULL: the call validates node ids and SYNCHRONISES (error on a bad id).
 *               Non-NULL: asynchronous; bit 0 is OR-ed in on a node id outside [0, N) (bit 1: level outside [0, L),
 *               mgv_build_level_lists) and the caller checks the word whenever it next synchronises.  Kernels stay
 *               memory-safe on bad input either way.
 */
size_t mgv_csr_workspace_bytes(int64_t N, int64_t E);
int mgv_build_csr(const int64_t* edge_index, int64_t E, int32_t N, const int32_t* code,
                  int32_t* in_ptr, int32_t* in_src, int32_t* out_ptr, int32_t* out_pack, int32_t* out_slot,
                  void* ws, size_t ws_bytes, int32_t* err_flag, mgv_stream_t stream);

/* ASAP level of every node == utils/dag_utils.py:10-37 top_sort(edge_index, N) (level 0 = no
 * predecessor, else 1 + max over predecessors).  reverse != 0 levelises the reversed graph
 * (return_order_info's backward_level, dag_utils.py:83-84): pass the out-CSR as the in-CSR and
 * vice versa.  info[0] = number of levels, info[1] = number of nodes levelised (< N means the
 * graph has a cycle; the reference would loop forever, this returns MGV_ERR_CYCLE after the
 * synchronising read-back).  SYNCHRONISES the stream (the caller needs the level count).
 */
size_t mgv_levelize_workspace_bytes(int64_t N);
int mgv_levelize(const int32_t* in_ptr, const int32_t* out_ptr, const int32_t* out_pack, int32_t N,
                 int32_t* level, int32_t* info_host, void* ws, size_t ws_bytes, mgv_stream_t stream);

/* Node lists per (level, code): order[N] = node ids stably sorted by (level, code) -- ascending
 * id inside a segment, i.e. G.forward_index[layer_mask & type_mask] (dg_ae_model_mig.py:89);
 * seg_ptr[L*MGV_NCODE + 1]; code_count_host[MGV_NCODE] = nodes of each code with level >= 1.
 * STREAMS: the circuits of a batch never exchange messages, so a batch may be cut into `streams` independent node sets
 * (stream_of_node int32 [N] in [0, streams), every edge inside one stream -- e.g. a partition of the batch's circuits; NULL
 * and streams = 1 otherwise).  The lists are then sorted by (stream, level, code): seg_ptr[streams*L*MGV_NCODE + 1], segment
 * (s, l, c) at index (s*L + l)*MGV_NCODE + c.  The level sweep runs the streams' level chains concurrently, each with its
 * own barrier; results do not depend on the cut.
 * SYNCHRONISES (returns the per-code counts used to size the persistent grids) -- unless code_count_host is NULL
 * and err_flag is given: then the caller supplies the counts itself (e.g. computed at collate time on the host,
 * where the reference computes forward_level, parser_func_others.py:63) and nothing synchronises.
 */
size_t mgv_level_lists_workspace_bytes(int64_t N, int32_t L);      /* pass streams * L */
int mgv_build_level_lists(const int32_t* level, const int32_t* code, const int32_t* stream_of_node, int32_t streams,
                          int32_t N, int32_t L, int32_t* order, int32_t* seg_ptr, int64_t* code_count_host,
                          void* ws, size_t ws_bytes, int32_t* err_flag, mgv_stream_t stream);

/* Row descriptors of the level sweep, in the order of `order` (32 bytes per row, so a tile's static schedule data is ONE
 * coalesced load instead of the chain order -> in_ptr -> in_src):
 *   desc[t] = { node = order[t], in_ptr[node], fan-in, out_ptr[node], fan-out, first three predecessors (in_src) or 0 }
 */
int mgv_build_sweep_desc(const int32_t* order, const int32_t* in_ptr, const int32_t* in_src, const int32_t* out_ptr,
                         int32_t N, int32_t* desc, mgv_stream_t stream);

/* Degree order of one CSR direction, for the tensor-core tiles of the struct encoder: order[N] = node ids sorted
 * by DESCENDING degree (degrees >= 255 tie), ascending id inside a degree, so the 128 rows of a tile have
 * near-equal fan-in/out and the gather lanes of a warp run the same trip count.  tile_cost[ntiles + 1], ntiles =
 * ceil(N / MGV_TILE_ROWS): exclusive prefix of (MGV_TILE_FIXED_COST + rows + neighbours + MGV_TILE_WAVE_COST * largest degree) per tile; persistent CTAs
 * take contiguous tile ranges of equal cost.
 * gdesc[N][4] (16-byte aligned): {node, first CSR slot, degree, first neighbour id} per row of the order.
 */
size_t mgv_degree_order_workspace_bytes(int64_t N);
/* The same gdesc / tile_cost for a degree order that already exists (e.g. built on the host when the batch was collated,
 * where the reference computes forward_level, parser_func_others.py:43-78): no sort, workspace as above. */
int mgv_build_degree_tiles(const int32_t* ptr, const int32_t* idx, const int32_t* order, int32_t N, int32_t* gdesc,
                           uint32_t* tile_cost, void* ws, size_t ws_bytes, mgv_stream_t stream);
int mgv_build_degree_order(const int32_t* ptr, const int32_t* idx, int32_t N, int32_t* order, int32_t* gdesc,
                           uint32_t* tile_cost, void* ws, size_t ws_bytes, mgv_stream_t stream);

/* ------------------------------------------------------------------ level sweep (fp32)
 * Replaces the level loop of Model.forward (dg_ae_model_mig.py:84-129 and the aig/xmg/xag
 * twins): per round, per level >= 1, per handled code: TFMlpAggr (arch/tfmlp.py:31-46) over the
 * predecessors' [hs || hf] rows, then the code's nn.GRU cell with h = hf[node], hf[node] <- h'.
 *
 * weights: the buffer mgv_sweep_pack fills (mgv_sweep_pack_bytes() bytes: natural blocks float [MGV_NCODE][MGV_SWEEP_PACK_FLOATS],
 * then the tensor-core weight images); handled_mask bit c set = code c has an aggregator/GRU pair.  rounds = 1 (the reference
 * default) runs on the tcgen05 kernels of csrc/sweep_tc.cu, rounds > 1 on the mma.sync kernels of csrc/sweep.cu.
 * Natural block layout (floats), D = 64:
 *      0  u[128]          = msg_k.weight^T attn_lin.weight[0,64:128]   (query part cancels in the softmax)
 *    128  WvT[128][64]    = msg_v.weight^T          8320 bv[64]
 *   8384  WihT[64][192]   = weight_ih_l0^T         20672 WhhT[64][192] = weight_hh_l0^T
 *  32960  bih[192]        33152 bhh[192]
 *  33344  Wv[64][128]     41536 Wih[192][64]       53824 Whh[192][64]          (natural copies, backward)
 * hf_all: float [R][N][64], zero-initialised by the caller; slot r = hf after round r.
 * sync: int32 [64] (grid barrier state of up to two streams; zeroed by the call).
 */
typedef struct mgv_schedule {
    int32_t N, L;
    int64_t E;
    const int32_t* order;      /* [N]   */
    const int32_t* seg_ptr;    /* [streams*L*MGV_NCODE+1] */
    const int32_t* in_ptr;     /* [N+1] */
    const int32_t* in_src;     /* [E]   */
    const int32_t* out_ptr;    /* [N+1] */
    const int32_t* out_pack;   /* [E]   */
    const int32_t* out_slot;   /* [E]   */
    int64_t code_count[MGV_NCODE];   /* host values: nodes per code at level >= 1 */
    const int32_t* deg_order_in;     /* [N] mgv_build_degree_order(in_ptr)   */
    const int32_t* deg_order_out;    /* [N] mgv_build_degree_order(out_ptr)  */
    const uint32_t* tile_cost_in;    /* [ceil(N/128)+1] */
    const uint32_t* tile_cost_out;
    const int32_t* gdesc_in;         /* [N][4] */
    const int32_t* gdesc_out;
    int32_t streams;                 /* independent node sets of the level lists (mgv_build_level_lists); 0 or 1 = one */
    int32_t reserved0;               /* 0 */
    const int32_t* sweep_desc;       /* [N][8] mgv_build_sweep_desc (needed by the single-round level sweep) */
} mgv_schedule;

/* precision (all compute entry points): MGV_PRECISION_FP32 = fp32-accurate tensor-core products (fp16 hi/lo planes, three
 * products, see csrc/mgv_tc.cuh), MGV_PRECISION_BF16 = one plane of bf16 operands with fp32 accumulation (tolerance 2e-2,
 * tests/test_gpu_parity.py::test_bf16_mode_within_stated_tolerance).  Storage stays fp32 in both.
 */
#define MGV_PRECISION_FP32 0
#define MGV_PRECISION_BF16 1
int mgv_level_sweep_fwd(const mgv_schedule* sch, int32_t rounds, uint32_t handled_mask,
                        const float* weights, const float* hs, float* hf_all,
                        int32_t* sync, int32_t precision, mgv_stream_t stream);

/* Backward of the sweep.  ghs [N][64] in/out: += d loss / d hs through every gather of every
 * round.  ghf [N][64] in/out: in = d loss / d hf (final round); clobbered.  grads: float
 * [MGV_NCODE][MGV_SWEEP_GRAD_FLOATS] out, natural layouts:
 *      0 du[128]   128 dWv[64][128]   8320 dbv[64]   8384 dWih[192][64]   20672 dWhh[192][64]
 *  32960 dbih[192]   33152 dbhh[192]
 * Workspace: mgv_sweep_bwd_workspace_bytes(N, E, grid) with grid = mgv_sweep_bwd_grid().
 */
int mgv_sweep_bwd_grid(void);
size_t mgv_sweep_bwd_workspace_bytes(int64_t N, int64_t E);
int mgv_level_sweep_bwd(const mgv_schedule* sch, int32_t rounds, uint32_t handled_mask,
                        const float* weights, const float* hs, const float* hf_all,
                        float* ghs, float* ghf, float* grads,
                        void* ws, size_t ws_bytes, int32_t* sync, int32_t precision, mgv_stream_t stream);

/* ------------------------------------------------------------------ struct encoder (fp32)
 * Replaces MultiGCNEncoder.forward (digae_layer.py:257-277) with AggConv (arch/gcn_conv.py:30-42):
 * state_0 = 1; per round: state <- LN(GRU([W sum_{in-nbrs} state + deg b || x], state)), then the
 * same over out-neighbours with aggr_r/update_r and the SAME LayerNorm.  num_enc encoders (source_conv,
 * target_conv of DirectMultiGCNEncoder, digae_layer.py:294-297) run batched over the same graph.
 *
 * weights: float [num_enc][2 dirs][MGV_STRUCT_PACK_FLOATS], host-prepared natural layouts with the AggConv
 * linear pre-composed into the GRU input weights (Wc = weight_ih_l0[:, :64] msg.weight, bc = weight_ih_l0[:, :64] msg.bias):
 *      0 Wcx[192][76]  cols 0..63 = Wc, cols 64..64+feat-1 = weight_ih_l0[:, 64:], rest 0
 *  14592 Whh[192][68]  weight_hh_l0, cols 64..67 = 0
 *  27648 bc[192]   27840 bih[192]   28032 bhh[192]   28224 ln_w[64]   28288 ln_b[64]   (pad to 28416)
 * x: float [N][feat] (feat <= MGV_MAX_FEAT).  states: float [num_enc][2][N][64] out, ping-pong slots: step k reads
 * slot (k-1)&1 and writes slot k&1 (slot 0 starts as ones, written by the call; after the last step it holds the encoder output).
 * tiles: NULL (inference) or mgv_struct_tiles_bytes(N, num_enc, rounds) bytes out: the [agg | h | x deg 1] tensor-core operand
 * tile of every step ([num_enc][2*rounds][ceil(N/128)][73728 bytes], fp16 hi/lo planes), which mgv_struct_encoder_bwd
 * recomputes from instead of gathering the neighbour sums a second time.
 */
size_t mgv_struct_fwd_workspace_bytes(int64_t N, int32_t num_enc);
size_t mgv_struct_tiles_bytes(int64_t N, int32_t num_enc, int32_t rounds);
int mgv_struct_encoder_fwd(const mgv_schedule* sch, int32_t num_enc, int32_t rounds, int32_t layernorm,
                           int32_t feat, const float* x, const float* weights, float* states, void* tiles,
                           void* ws, size_t ws_bytes, int32_t precision, mgv_stream_t stream);
/* tiles: the operand tiles mgv_struct_encoder_fwd saved (required).  gout: float [num_enc][N][64] = d loss / d (encoder
 * output).  grads: float [num_enc][2][MGV_STRUCT_GRAD_FLOATS] out, SAME layout as the weight block (d Wcx, d Whh, d bc,
 * d bih, d bhh, d ln_w, d ln_b; padding columns are zero).  The host maps d Wc / d bc back to msg.* and weight_ih_l0. */
size_t mgv_struct_bwd_workspace_bytes(int64_t N, int32_t num_enc);
int mgv_struct_encoder_bwd(const mgv_schedule* sch, int32_t num_enc, int32_t rounds, int32_t layernorm,
                           int32_t feat, const float* x, const float* weights, const void* tiles,
                           const float* gout, float* grads, void* ws, size_t ws_bytes,
                           int32_t precision, mgv_stream_t stream);

/* ------------------------------------------------------------------ fused reparam + KL + func loss
 * Replaces DirectedGVAE.sample's elementwise part (digvae_model.py:138-141), the KL of
 * trainer.py:145-148 and the truth-table-similarity loss of trainer.py:157-163 with
 * zero_normalization (utils/utils.py:32-36) in ONE launch.
 *   mu/logstd/eps: float [2][N][64] (s then t); z out [2][N][64]          (N may be 0: VAE part skipped)
 *   hf float [Nf][64]; pair int64 [2][P]; tt_sim float [P]                 (P may be 0: func part skipped)
 *   out float [8]: 0 kl, 1 func_loss, 2 mean(dis), 3 std(dis), 4 mean(tt), 5 std(tt), 6 sum g*zd, 7 mean g
 *   ws: float/double scratch, mgv_vae_func_workspace_bytes(P), zero-initialised by the caller.
 */
size_t mgv_vae_func_workspace_bytes(int64_t P);
int mgv_vae_func_loss_fwd(const float* mu, const float* logstd, const float* eps, float* z, int64_t N,
                          const float* hf, const int64_t* pair, const float* tt_sim, int64_t P,
                          float* out, void* ws, size_t ws_bytes, mgv_stream_t stream);
/* g_out float [2] on device: d L / d kl, d L / d func_loss; gz float [2][N][64] = d L / d z.
 * gmu, glogstd out [2][N][64]; ghf [Nf][64] in/out: func-loss gradient is atomically ADDED. */
int mgv_vae_func_loss_bwd(const float* g_out, const float* gz, const float* mu, const float* logstd,
                          const float* eps, float* gmu, float* glogstd, int64_t N,
                          const float* hf, const int64_t* pair, const float* tt_sim, int64_t P,
                          const float* out, const void* ws, float* ghf, mgv_stream_t stream);

/* ------------------------------------------------------------------ parameter packing (host pointer tables -> weight blocks)
 * `params` are HOST arrays of DEVICE pointers to the reference modules' fp32 parameters (contiguous, natural shapes).
 * struct encoder, per encoder: [aggr.msg.weight, aggr.msg.bias, update.weight_ih_l0, update.weight_hh_l0, update.bias_ih_l0,
 *   update.bias_hh_l0, the same six of aggr_r / update_r, (ln.weight, ln.bias if layernorm)]  ->  pack [num_enc][2][MGV_STRUCT_PACK_FLOATS].
 * mgv_struct_unpack_grads applies the chain rule of the composition (Wc = W_ih[:, :64] W_msg, bc = W_ih[:, :64] b_msg) to the gradient
 * blocks and writes, per encoder, d(those parameters) back to back in the same order and natural shapes.
 * level sweep, per listed gate code: [attn_lin.weight, msg_k.weight, msg_v.weight, msg_v.bias, weight_ih_l0, weight_hh_l0,
 *   bias_ih_l0, bias_hh_l0]  ->  pack: a buffer of mgv_sweep_pack_bytes() bytes = the natural blocks [MGV_NCODE][MGV_SWEEP_PACK_FLOATS]
 *   followed by one tensor-core weight image per code (Wc = weight_ih_l0 msg_v.weight as fp16 hi/lo -- bf16 for precision 1 --
 *   planes in the UMMA layout + composed biases, csrc/sweep_layout.cuh); blocks / images of unlisted codes are untouched.
 *   This buffer is the `weights` argument of mgv_level_sweep_fwd / _bwd.
 * mgv_sweep_unpack_grads writes per listed code d attn_lin.weight [128] then d msg_k.weight [64][128]; the other gradients are
 * read in place from the gradient block (natural layouts).
 */
int mgv_struct_pack(const void* const* params, int32_t num_enc, int32_t layernorm, int32_t feat, float* pack, mgv_stream_t stream);
int mgv_struct_unpack_grads(const void* const* params, int32_t num_enc, int32_t layernorm, int32_t feat,
                            const float* grads, float* out, mgv_stream_t stream);
size_t mgv_sweep_pack_bytes(void);
int mgv_sweep_pack(const void* const* params, const int32_t* codes, int32_t n, float* pack, int32_t precision, mgv_stream_t stream);
int mgv_sweep_unpack_grads(const void* const* params, const int32_t* codes, int32_t n, const float* grads, float* out,
                           mgv_stream_t stream);

/* ------------------------------------------------------------------ reconstruction loss + negative sampler
 * Replaces Model.recon_loss (dg_ae_model_mig.py:169-191) around the directed inner-product decoder
 * (digae_layer.py:26-33): st = hs_decompose(hs) = [s | t] float [N][128]; value(u -> v) = sigmoid(s_u . t_v);
 *   out float [3]: loss = -mean_pos log(value + 1e-15) - mean_neg log(1 - value + 1e-15), its pos part, its neg part
 *   sig float [Ep + En], pred int32 [Ep + En] (value > 0.5), positives first  (pred_bin of the reference)
 *   pos int64 [2][Ep], neg int64 [2][En]; ws >= 16 bytes; err_flag: bit 2 OR-ed in on an edge end outside [0, N).
 * mgv_negative_sample stands in for torch_geometric.utils.negative_sampling (dg_ae_model_mig.py:177-180): `count`
 * ordered pairs (u, v), u != v, not an edge u -> v of the out-CSR, drawn by rejection from a counter-based hash of `seed`.
 */
int mgv_negative_sample(const int32_t* out_ptr, const int32_t* out_pack, int32_t N, int64_t count, uint64_t seed,
                        int64_t* neg, mgv_stream_t stream);
/* The per-batch edge "split" of the training loop with val_ratio = test_ratio = 0 (preprocessing.py:8-83 as called at
 * trainer.py:133: every edge is a training edge, in random order; the reference's N x N mask is unused there and is not
 * built).  out int64 [2][E] = edge_index[:, pi], pi a pseudo-random permutation keyed by `seed` (4-round Feistel network with
 * cycle walking: one launch, O(E), no sort).  out must not alias edge_index. */
int mgv_permute_edges(const int64_t* edge_index, int64_t E, uint64_t seed, int64_t* out, mgv_stream_t stream);
int mgv_recon_loss_fwd(const float* st, int32_t N, const int64_t* pos, int64_t Ep, const int64_t* neg, int64_t En,
                       float* out, float* sig, int32_t* pred, void* ws, size_t ws_bytes, int32_t* err_flag,
                       mgv_stream_t stream);
/* g_loss: device float = d L / d loss; gst float [N][128] zero-initialised by the caller, gradients are atomically added. */
int mgv_recon_loss_bwd(const float* st, int32_t N, const int64_t* pos, int64_t Ep, const int64_t* neg, int64_t En,
                       const float* sig, const float* g_loss, float* gst, mgv_stream_t stream);

/* ------------------------------------------------------------------ fused readout head (probability MLP + clamp + L1 loss)
 * Replaces Model.pred_prob's MLP(64, 32, 1, num_layer = 3, p_drop, batchnorm, relu) (dg_ae_model_mig.py:44, arch/mlp.py:14-56), the
 * clamp to [0, 1] (dg_ae_model_mig.py:150-152) and nn.L1Loss of trainer.py:154-156: forward ONE launch, backward ONE launch.
 *   params: HOST array of 14 DEVICE pointers, fp32: fc.0.weight [32][64], fc.0.bias, bn1.weight, bn1.bias, bn1.running_mean,
 *           bn1.running_var, fc.4.weight [32][32], fc.4.bias, bn2.weight, bn2.bias, bn2.running_mean, bn2.running_var,
 *           fc.8.weight [1][32], fc.8.bias.  training != 0: batch statistics (biased variance), running statistics updated in
 *           place with `momentum` (unbiased variance), dropout with keep probability 1 - p_drop from a counter-based hash of
 *           (seed, node, layer, channel); training == 0: running statistics, no dropout.
 *   x float [N][64]; target float [N] or NULL; pred float [N] out = clamp(mlp(x), 0, 1); loss float [1] out = mean |pred - target|
 *   saved float [N][64] out (pre-normalisation activations), stats float [128] out (mean / 1 / std of both BatchNorms): for the backward
 *   mask uint32 [N][2] out or NULL: keep bits of the two dropout layers (bit c = channel c kept), for tests
 *   sync int32 [1] (grid barrier, zeroed by the call); ws >= mgv_readout_workspace_bytes(N)
 * Backward: g_pred float [N] or NULL (d L / d pred), g_loss device float or NULL (d L / d loss); gx float [N][64] out;
 *   grads float [3297] out: d fc.0.weight 2048 | d fc.0.bias 32 | d bn1.weight 32 | d bn1.bias 32 | d fc.4.weight 1024 | d fc.4.bias 32 |
 *   d bn2.weight 32 | d bn2.bias 32 | d fc.8.weight 32 | d fc.8.bias 1.  Same seed / p_drop / training as the forward.
 */
size_t mgv_readout_workspace_bytes(int64_t N);
int mgv_readout_fwd(const float* x, int64_t N, const void* const* params, int32_t training, float p_drop, uint64_t seed,
                    float momentum, float eps, const float* target, float* pred, float* loss, float* saved, float* stats,
                    uint32_t* mask, void* ws, size_t ws_bytes, int32_t* sync, mgv_stream_t stream);
int mgv_readout_bwd(const float* x, int64_t N, const void* const* params, int32_t training, float p_drop, uint64_t seed,
                    const float* target, const float* saved, const float* stats, const float* g_pred, const float* g_loss,
                    float* gx, float* grads, void* ws, size_t ws_bytes, int32_t* sync, mgv_stream_t stream);

/* ------------------------------------------------------------------ tensor-core self test (diagnostic)
 * One 128-row tcgen05 tile product through the operand layouts / descriptors / fp16 hi-lo split the kernels
 * use (csrc/mgv_tc.cuh).  D is fp32 row-major.
 *   mode 0: D[128][N]  = A[128][K] . B[N][K]^T                K in {64,128}     (K-major SW128 operands)
 *   mode 1: D[128][N]  = A[128 rows][128]^T . B[128 rows][N]  N % 64 == 0       (both read MN-major: weight-gradient form)
 *   mode 2: D[128][N]  = A[128][16] . B[N][16]^T                                (plain 16-column tiles)
 *   mode 3: D[128][16] = A[128 rows][128]^T . B[128 rows][16]                   (MN-major SW128 x MN-major plain)
 *   mode 4: D[128][64] = A[128][192] . B[192][64]                               (K-major x MN-major: data-gradient form)
 *   mode 5: D[128][128] = A[128][64] . B[64][128]      A written to TENSOR MEMORY (tcgen05.st), B MN-major from two
 *           64-column blocks: the data-gradient product of the struct-encoder backward (struct_bwd_tc.cu)
 */
/* ------------------------------------------------------------------ small Linear layers around the path
 * Weight / bias gradient of y = x W^T + b for the nn.Linear layers whose input is one row per node: hs_linear,
 * hs_decompose (dg_ae_model_mig.py:46-47) and the readout MLP (arch/mlp.py:14-56):
 *     dW[O][I] = sum_n gy[n][O] x[n][I],  db[O] = sum_n gy[n][O]   (db may be NULL),  1 <= I, O <= 128, fp32, deterministic.
 * Replaces torch.autograd's AddmmBackward weight GEMM, which a library runs as one output tile on one SM with K = N.
 */
size_t mgv_linear_wgrad_workspace_bytes(int64_t N, int32_t I, int32_t O);
int mgv_linear_wgrad(const float* x, const float* gy, int64_t N, int32_t I, int32_t O, float* dW, float* db,
                     void* ws, size_t ws_bytes, mgv_stream_t stream);

/* Forward and data gradient of the same layers on the tensor cores (csrc/linear_tc.cu; fp16 hi/lo planes, fp32-accurate):
 *     out[N][P] = in[N][Q] . M[P][Q]^T (+ bias[P]),  P, Q in {64, 128}
 *   transposed = 0: M = W, W given as [P][Q]  (y = x W^T + b: P = out features, Q = in features)
 *   transposed = 1: M = W^T, W given as [Q][P]  (gx = gy W: P = in features, Q = out features; bias NULL)
 * Replaces torch.addmm / AddmmBackward's data GEMM (cuBLAS fp32 SIMT, 37 us at N = 65 818) for hs_linear, hs_decompose and the
 * four Linear layers of DirectedGVAE.sample (digvae_model.py:105-142).
 */
int mgv_linear_tc(const float* in, int64_t N, const float* W, const float* bias, int32_t P, int32_t Q, int32_t transposed,
                  float* out, mgv_stream_t stream);

int mgv_tc_selftest(int32_t mode, const float* A, const float* B, float* D, int32_t K, int32_t N, mgv_stream_t stream);

/* ------------------------------------------------------------------ logic simulation (labels: signal probability, truth-table distance)
 * Bit-parallel simulation of the batch under 64 input patterns per uint64 word, level by level over the schedule's
 * (stream, level, code) lists (any `streams`).  What the reference's dataset tooling produces as `prob` and `tt_dis`.
 *   fn_table_host int32 [MGV_NCODE], HOST: gate function of each code; MGV_FN_NONE marks a code the circuit kind lacks.
 *     AIG: {INPUT, AND, NOT};  MIG / XMG / XAG (gate_to_index, parser.py:133): {INPUT, MAJ, NOT, AND, OR, XOR}.
 *     AND, OR and XOR reduce over all predecessors (fan-in >= 2); NOT has fan-in 1, MAJ fan-in 3, INPUT fan-in 0.
 *   code int32 [N] raw gate codes; level int32 [N] the schedule's levels.
 * mgv_logic_sim_validate SYNCHRONISES and returns MGV_ERR_ARG naming the first bad node (undefined code, INPUT with
 * predecessors, gate with fan-in 0, NOT / MAJ / AND / OR / XOR with the wrong fan-in, a predecessor not at a lower
 * level), else the first pair with an id outside [0, N).  pairs int64 [2][P].  ws >= 16 bytes.  Run it before any pass:
 * the pass assumes a valid circuit (and stays memory-safe, with meaningless counts, on an undefined code).
 * mgv_logic_sim_pass simulates words [first_word, first_word + W) of every node:
 *   mode MGV_SIM_RANDOM:     word w of an INPUT = mix(mix(seed) ^ (rank << 40 | w)), mix = the splitmix64 finaliser;
 *   mode MGV_SIM_EXHAUSTIVE: pattern t = 64 w + bit, the INPUT takes bit `rank` of t;
 *   input_rank int32 [N]: an INPUT's position among the INPUTs of its own circuit (other entries are not read);
 *   sim: mgv_logic_sim_bytes(N, W) bytes, 32-byte aligned, scratch ([N][W rounded up to 4] words; INPUT words included);
 *   ones uint64 [N] in/out: += patterns of the pass where node v is 1;
 *   diff uint64 [P] in/out: += patterns of the pass where the two nodes of pair p differ (pairs / diff NULL when P = 0).
 * Counts are integers, so the result is deterministic and independent of how the words are split into passes.
 */
#define MGV_FN_NONE 0
#define MGV_FN_INPUT 1
#define MGV_FN_AND 2
#define MGV_FN_OR 3
#define MGV_FN_XOR 4
#define MGV_FN_NOT 5
#define MGV_FN_MAJ 6
#define MGV_SIM_RANDOM 0
#define MGV_SIM_EXHAUSTIVE 1
size_t mgv_logic_sim_bytes(int64_t N, int32_t W);
int mgv_logic_sim_validate(const mgv_schedule* sch, const int32_t* code, const int32_t* level,
                           const int32_t* fn_table_host, const int64_t* pairs, int64_t P,
                           void* ws, size_t ws_bytes, mgv_stream_t stream);
int mgv_logic_sim_pass(const mgv_schedule* sch, const int32_t* code, const int32_t* input_rank,
                       const int32_t* fn_table_host, int32_t mode, uint64_t seed, int64_t first_word, int32_t W,
                       uint64_t* sim, uint64_t* ones, const int64_t* pairs, int64_t P, uint64_t* diff,
                       mgv_stream_t stream);

#define MGV_OK 0
#define MGV_ERR_ARG (-1)
#define MGV_ERR_CUDA (-2)
#define MGV_ERR_WORKSPACE (-3)
#define MGV_ERR_CYCLE (-4)

#ifdef __cplusplus
}
#endif
#endif /* MGV_B200_H */
