"""Dev tool: per-phase clock64 trace of one backward step kernel (step k = 2)."""
import os, sys, ctypes
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "multi-gate-vae_b200"), ROOT]
import torch, bench, deepgate
from deepgate import _native as nat
w = bench.WORKLOADS[sys.argv[1] if len(sys.argv) > 1 else "cfg2"]
dev = torch.device("cuda", 0)
enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=4, t_rounds=4, layernorm=True).to(dev)
G = bench.make_host_batch(w, 0, 0).copy_to(dev, non_blocking=False)
feat = torch.nn.functional.one_hot(G.x[:, 1].to(torch.int64), num_classes=6).to(torch.float32)
lib = nat.lib()
lib.mgv_debug_set_trace.argtypes = [ctypes.c_void_p]
for i in range(2):
    s, t = enc(feat, feat, G.edge_index); (s.sum() + t.sum()).backward()
s, t = enc(feat, feat, G.edge_index)
tr = torch.zeros(2 * 74 * 16 * 16, dtype=torch.int64, device=dev)
lib.mgv_debug_set_trace(ctypes.c_void_p(tr.data_ptr()))
(s.sum() + t.sum()).backward()
torch.cuda.synchronize()
lib.mgv_debug_set_trace(ctypes.c_void_p(0))
t = tr.view(2 * 74, 16, 16).cpu().double()
if os.environ.get("MGV_TRACE_WGRAD"):
    spans = [("producer: wait stage empty", 0, 1), ("stage: copies issued -> landed", 1, 2), ("rescale + hand-over", 2, 3),
             ("MMA: wait ready", 4, 5), ("MMA: issue", 5, 6)]
    valid = (t[:, :, 0] > 0) & (t[:, :, 6] > 0)
    for n, a, b in spans:
        d = (t[:, :, b] - t[:, :, a])[valid]
        print("%-46s mean %7.0f  med %7.0f  max %7.0f cycles" % (n, d.mean(), d.median(), d.max()))
    per = (t[:, 1:, 5] - t[:, :-1, 5])[valid[:, 1:] & valid[:, :-1]]
    print("stage period mean %.0f cycles" % per.mean())
    v0 = t[:, 0, 10] > 0
    print("first copy -> flush start %.0f, wait done %.0f, flush %.0f cycles" % ((t[:, 0, 8] - t[:, 0, 0])[v0].mean(), (t[:, 0, 9] - t[:, 0, 8])[v0].mean(), (t[:, 0, 10] - t[:, 0, 9])[v0].mean()))
else:
    # tcgen05 pointwise kernel (struct_bwd_tc.cu): slots 3-12 epilogue thread 0, 13-15 slowest gather warp
    t = torch.cat([t, torch.cat([t[:, 1:, 4:5], torch.zeros(t.shape[0], 1, 1, dtype=t.dtype)], 1)], 2)      # slot 16 = next tile's slot 4
    spans = [("pass 1 + LayerNorm statistics", 4, 5), ("pass 2 (LN + GRU backward)", 5, 12), ("tile scale (amax, barrier)", 12, 6),
             ("pass 3 (planes -> TMEM + HBM) + barrier", 6, 7), ("MMA issue: data gradient + next recompute (thread 0)", 7, 3),
             ("data-gradient MMAs (planes ready -> done)", 7, 8), ("output stores", 8, 9),
             ("tile end -> next tile's accumulators ready", 9, 16),
             ("gather: d state rows + neighbour sums (slowest warp)", 13, 14), ("gather: wait g_empty + store", 14, 15)]
    valid = (t[:, :, 4] > 0) & (t[:, :, 9] > 0) & (t[:, :, 16] > 0) & (t[:, :, 3] > 0)
    for n, a, b in spans:
        d = (t[:, :, b] - t[:, :, a])[valid]
        print("%-56s mean %7.0f  med %7.0f  max %7.0f cycles" % (n, d.mean(), d.median(), d.max()))
    d = (t[:, :, 16] - t[:, :, 4])[valid]
    print("tile period mean %.0f cycles (n=%d)" % (d.mean(), d.numel()))
