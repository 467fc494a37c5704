"""Dev tool: time the struct encoder forward / backward calls alone (CUDA events), cfg given on the command line."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "multi-gate-vae_b200"), ROOT]
import torch, bench, deepgate
w = bench.WORKLOADS[sys.argv[1] if len(sys.argv) > 1 else "cfg2"]
dev = torch.device("cuda", 0)
enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=4, t_rounds=4, layernorm=True).to(dev)
G = bench.make_host_batch(w, 0, 0).copy_to(dev, non_blocking=False)
feat = torch.nn.functional.one_hot(G.x[:, 1].to(torch.int64), num_classes=6).to(torch.float32)
def run(n):
    tf = tb = 0.0
    for i in range(n):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record(); s, t = enc(feat, feat, G.edge_index); l = s.sum() + t.sum(); e[1].record(); l.backward(); e[2].record()
        torch.cuda.synchronize(); tf += e[0].elapsed_time(e[1]); tb += e[1].elapsed_time(e[2])
    return tf / n, tb / n
run(3)
f, b = run(10)
print("N=%d E=%d  struct fwd %.3f ms  bwd %.3f ms  (chunk=%s)" % (G.x.size(0), G.edge_index.size(1), f, b,
      os.environ.get("MGV_STRUCT_CHUNK", "default")))
