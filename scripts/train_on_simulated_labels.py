"""Do simulated labels carry signal the model can learn?

    python scripts/train_on_simulated_labels.py [--circuits 600] [--epochs 30] [--seed 0]

Labels synthetic MIG circuits (synth's "mig4" mix: MAJ, NOT, AND, OR) by logic simulation on cuda:0
(deepgate.label_circuits), trains the DG_AE MIG model with ``Trainer`` for a fixed, seeded number of epochs on 90 % of them,
and prints the held-out prob L1 of the model next to the held-out L1 of the best constant predictor (the median of the training labels).  Only numbers are reported: no threshold
has been established.  The pure MAJ / NOT mix is not used: MAJ and NOT of balanced inputs stay balanced, so its labels sit
within about 0.01 of 0.5 and a constant predicts them almost exactly.
"""
import argparse
import json
import os
import sys
import tempfile
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "multi-gate-vae_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def held_out_l1(model, dataset, device):
    import deepgate
    model.eval()
    err, count = 0.0, 0
    with torch.no_grad():
        for batch in deepgate.DataLoader(dataset, batch_size=32):
            batch = batch.to(device)
            _, hf = model(batch)
            pred = model.pred_prob(hf).reshape(-1)
            err += float((pred - batch.prob.reshape(-1)).abs().sum())
            count += pred.numel()
    return err / count


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--circuits", type=int, default=600)
    ap.add_argument("--epochs", type=int, default=30)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import deepgate
    from deepgate import synth
    torch.manual_seed(args.seed)
    circuits = synth.make_circuits("mig4", args.circuits, (8, 24), (40, 300), cfg=900 + args.seed)
    for c in circuits:
        c.pop("tt_pair_index")                                  # drawn anew by label_circuits (distinct nodes)
    labelled = deepgate.label_circuits(circuits, "mig", "cuda:0", n_pairs=64, seed=args.seed)
    graphs = [deepgate.parse_pyg_mlpgate(c["x"], c["edge_index"], c["prob"], c["tt_sim"], c["tt_pair_index"]) for c in labelled]
    cut = int(0.9 * len(graphs))
    train, val = deepgate.CircuitDataset(graphs[:cut]), deepgate.CircuitDataset(graphs[cut:])
    train_prob = np.concatenate([c["prob"] for c in labelled[:cut]])
    val_prob = np.concatenate([c["prob"] for c in labelled[cut:]])
    const = float(np.median(train_prob))
    const_l1 = float(np.abs(val_prob - const).mean())
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=1, t_rounds=1)
    model = deepgate.dg_ae_model_mig.Model(struct_encoder=enc, dim_hidden=64)
    with tempfile.TemporaryDirectory() as tmp:
        trainer = deepgate.Trainer(types.SimpleNamespace(model="DG_AE", type="mig"), model, training_id="simlabels",
                                   save_dir=tmp, device="cuda:0", batch_size=32, distributed=False, lr=args.lr,
                                   rc_prob_func_weight=[1.0, 4.0, 2.0])
        before = held_out_l1(trainer.model, val, "cuda:0")
        trainer.train(args.epochs, train, val)
        after = held_out_l1(trainer.model, val, "cuda:0")
    rec = {"circuits": len(labelled), "train": cut, "held_out": len(graphs) - cut, "held_out_nodes": int(val_prob.size),
           "epochs": args.epochs, "seed": args.seed, "lr": args.lr, "held_out_prob_l1_untrained": round(before, 4),
           "held_out_prob_l1_trained": round(after, 4), "held_out_prob_l1_best_constant": round(const_l1, 4),
           "best_constant": round(const, 4), "card": torch.cuda.get_device_name(0)}
    print(json.dumps(rec))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "train_on_simulated_labels.json"), "w") as f:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
