#!/usr/bin/env python
"""Benchmark of the level-synchronous DAG message-passing path (BASELINE.json metric:
gates/s propagated fwd+bwd, all rounds, and train-step ms).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one training step of the reference's loop on one synthetic batch: Model.forward(G)
(level schedule + struct encoder + level sweep), recon / prob / func losses, backward, gradient
all-reduce (N > 1) and Adam.  ``value`` = gates propagated per second over all ranks with the
batches resident in HBM; ``e2e`` = the same through Trainer.train_step with the batch in pinned
HOST memory (H2D copy and loss read-back inside the timed region).  ``--impl reference`` times the
reference algorithm's CPU restatement (oracle/dg_oracle.py, per-node ``subgraph`` loop included)
on the host cores -- the one other place this file executes oracle/.  ``--dump-outputs DIR`` writes
what ``Trainer.train_step`` returned in the last timed step of ``value`` (losses, hs, hf, link
predictions) as float32 ``DIR/<name>.npy``.  The same arguments give the same inputs in every run --
the batches, the seeded weights (Adam runs at learning rate 0, see measure) and torch's seed for the
step's random draws -- so two builds can be compared output for output.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "multi-gate-vae_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: kind, gate mix, circuits per GPU, n_pi, n_gates, window, sweep rounds   (SURVEY.md section 8d)
    "cfg1": dict(kind="mig", mix="mig4", batch=4, n_pi=16, n_gates=200, window=None, rounds=1, cfg=1),
    "cfg2": dict(kind="aig", mix="aig", batch=64, n_pi=(16, 64), n_gates=(500, 1500), window=None, rounds=1, cfg=2),
    "cfg3-xmg": dict(kind="xmg", mix="xmg", batch=64, n_pi=(16, 64), n_gates=(500, 1500), window=None, rounds=2, cfg=3),
    "cfg3-xag": dict(kind="xag", mix="xag", batch=64, n_pi=(16, 64), n_gates=(500, 1500), window=None, rounds=2, cfg=3),
    "cfg4": dict(kind="xmg", mix="xmg", batch=64, n_pi=(16, 64), n_gates=(500, 1500), window=None, rounds=1, cfg=4,
                 variational=True, precision="bf16"),
    "cfg5-k1": dict(kind="mig", mix="mig", batch=1, n_pi=16, n_gates=100000, window=880, rounds=1, cfg=5),
    "cfg5-k8": dict(kind="mig", mix="mig", batch=8, n_pi=16, n_gates=100000, window=880, rounds=1, cfg=5),
    "cfg5-k64": dict(kind="mig", mix="mig", batch=64, n_pi=16, n_gates=100000, window=880, rounds=1, cfg=5),
}
HANDLED = {"aig": (1, 2), "mig": (1, 2, 3, 4), "xmg": (1, 2, 3, 4, 5), "xag": (2, 3, 5)}
LOSS_W = (1.0, 4.0, 4.0)      # stage-3 weights of the reference schedule (train.py:91)
DUMP_BYTES = 60 * 10 ** 6     # --dump-outputs: data bytes of one dump, under 64 MB with the .npy headers


def write_outputs(out_dir, arrays):
    """``arrays`` (name -> CPU tensor) as float32 ``out_dir/<name>.npy``.  Above DUMP_BYTES in all, every array of more than one
    row keeps the same share of its rows, drawn with a fixed seed (arrays of the same length keep the same rows), and
    ``<name>_rows.npy`` (float64) lists the rows kept."""
    os.makedirs(out_dir, exist_ok=True)
    multi = {k for k, a in arrays.items() if a.dim() > 0 and a.shape[0] > 1}
    fixed = sum(4 * a.numel() for k, a in arrays.items() if k not in multi)
    per_share = sum(a.shape[0] * (4 * a[0].numel() + 8) for k, a in arrays.items() if k in multi)
    share = min(1.0, (DUMP_BYTES - fixed) / max(per_share, 1))
    for name, a in sorted(arrays.items()):
        a = a.float()
        if share < 1.0 and name in multi:
            rows = torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:max(1, int(a.shape[0] * share))]
            rows = rows.sort().values
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.double().numpy())
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def make_host_batch(w, rank, idx, own_sizes=False):
    import deepgate
    from deepgate import synth
    # ranks draw different circuits of the SAME sizes (size-bucketed sampler): weak scaling without size skew between ranks.
    # own_sizes: every rank also draws its own circuit SIZES (the reference's plain DistributedSampler, trainer.py:179-192).
    circuits = synth.make_circuits(w["mix"], w["batch"], w["n_pi"], w["n_gates"],
                                   cfg=w["cfg"] + 100 * rank + 10 * idx, window=w["window"],
                                   size_cfg=w["cfg"] + 10 * idx + (1000 * rank if own_sizes else 0))
    return deepgate.circuits_to_batch(circuits)


def batch_stats(b, kind):
    code = b.gate.reshape(-1).long()
    lvl = b.forward_level.long()
    indeg = torch.bincount(b.edge_index[1], minlength=code.numel())
    handled = torch.zeros_like(code, dtype=torch.bool)
    for c in HANDLED[kind]:
        handled |= code == c
    live = handled & (lvl >= 1)
    d = indeg[live].double()
    n, e = code.numel(), b.edge_index.size(1)
    return {
        "N": n, "E": e, "L": int(lvl.max()) + 1, "gates": int(live.sum()),
        # algorithmic bytes, SURVEY.md section 8d (fp32): fwd 516 d + 520, bwd 1540 d + 776 per gate
        "sweep_fwd_bytes": float((516 * d + 520).sum()), "sweep_bwd_bytes": float((1540 * d + 776).sum()),
        # struct encoder per half-step launch, both encoders: fwd 256 (deg + 2), bwd 256 (3 deg + 3) per node
        "struct_fwd_bytes": 2.0 * 256 * (e + 2 * n), "struct_bwd_bytes": 2.0 * 256 * (3 * e + 3 * n),
    }


class ClockSampler(object):
    """nvidia-smi polled every 25 ms from before the warm-up until after the timed region (its start-up alone can take
    longer than a short timed region); only the samples whose timestamps fall inside [mark_begin, mark_end] are used."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.index = index
        self.t0 = self.t1 = None

    def start(self):
        if os.environ.get("MGV_BENCH_NO_SAMPLER"):
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        import datetime
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if self.t0 is not None and self.t1 is not None and not (self.t0 - 0.03 <= ts <= self.t1 + 0.03):
                    continue
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nme, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.path)
        top = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": statistics.median(top) if top else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------- reference arm (CPU)
def cpu_step(kind, P, host_batch, rounds, n_sample):
    """One train step of the reference algorithm (oracle port) on the first ``n_sample`` circuits."""
    from oracle import dg_oracle as O
    ptr = host_batch.ptr.tolist()
    n = ptr[n_sample]
    emask = host_batch.edge_index[1] < n
    ei = host_batch.edge_index[:, emask]
    pmask = (host_batch.tt_pair_index[0] < n) & (host_batch.tt_pair_index[1] < n)
    g = torch.Generator().manual_seed(0)
    G = {"code": host_batch.gate.reshape(-1).long()[:n], "edge_index": ei, "forward_level": host_batch.forward_level[:n],
         "prob": host_batch.prob[:n], "tt_pair_index": host_batch.tt_pair_index[:, pmask], "tt_sim": host_batch.tt_sim[pmask],
         "train_pos_edge_index": ei[:, torch.randperm(ei.size(1), generator=g)],
         "neg_edge_index": torch.randint(0, n, (2, ei.size(1)), generator=g)}
    for p in P.values():
        if p.requires_grad:
            p.grad = None
    t0 = time.perf_counter()
    total, _ = O.train_step_losses(P, kind, G, LOSS_W, rounds, literal_subgraph=True)
    total.backward()
    dt = time.perf_counter() - t0
    code, lvl = G["code"], G["forward_level"]
    handled = torch.zeros_like(code, dtype=torch.bool)
    for c in HANDLED[kind]:
        handled |= code == c
    return dt, int((handled & (lvl >= 1)).sum()) * rounds


def cpu_params(kind):
    from oracle import dg_oracle as O
    P = O.synth_state_dict(kind, 2)
    for k, p in P.items():
        p.requires_grad_("running" not in k)
    return P


def pick_sample(w, budget_s=20.0):
    """Circuits in the CPU sample.  The reference's per-node subgraph loop costs ~ nodes * edges compares;
    calibrated on 8 Xeon cores: 64 x ~1000-gate circuits -> 17.5 s per train step (c = 4.3e-9 s / node^2)."""
    per = (w["n_gates"] if isinstance(w["n_gates"], int) else sum(w["n_gates"]) / 2)
    if per >= 50000:
        return 1
    return max(1, min(w["batch"], int((budget_s / 4.3e-9) ** 0.5 / per)))


def run_reference(args, w):
    """The reference's CPU path (oracle port with the reference's literal per-node ``subgraph`` loop) on the host cores, on the
    SAME batch the B200 arm times.  Every timed step runs the full batch when the whole run then fits the time budget
    (calibrated by one untimed full-batch step); otherwise the first steps are the full batch and the rest a bounded sample,
    and ``sample`` says so."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    hb = make_host_batch(w, 0, 0)
    P = cpu_params(w["kind"])
    full = w["batch"]
    quarter = max(1, full // 4)
    for _ in range(max(args.warmup - 1, 0)):              # warm-up: quarter batches, then ONE full batch that calibrates the budget
        cpu_step(w["kind"], P, hb, w["rounds"], quarter)
    est_full, _g = cpu_step(w["kind"], P, hb, w["rounds"], full)
    budget = float(os.environ.get("MGV_REF_BUDGET_S", 240.0))
    n_full = max(1, min(args.steps, int(budget / max(est_full, 1e-3))))
    ns_rest = full if n_full == args.steps else pick_sample(w, max(1.0, (budget - n_full * est_full) / max(args.steps - n_full, 1)))
    tot_t, tot_g = 0.0, 0
    for i in range(args.steps):
        dt, gates = cpu_step(w["kind"], P, hb, w["rounds"], full if i < n_full else ns_rest)
        tot_t += dt
        tot_g += gates
    val = tot_g / tot_t
    sample = "%d of %d timed steps on the full batch of %d circuits%s; oracle port, per-node subgraph loop as in the reference" % (
        n_full, args.steps, full, "" if n_full == args.steps else ", the rest on %d circuits" % ns_rest)
    st = batch_stats(hb, w["kind"])
    print(json.dumps({
        "impl": "reference", "metric": "gates_per_s_fwd_bwd", "value": val, "unit": "gates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "model": "DG_AE-" + w["kind"], "circuits_per_gpu": w["batch"],
                   "nodes_per_gpu": float(st["N"]), "edges_per_gpu": float(st["E"]), "levels": float(st["L"]),
                   "sweep_rounds": w["rounds"], "s_rounds": 4, "t_rounds": 4, "layernorm": True, "dim_hidden": 64,
                   "step": "forward + recon/prob/func losses + backward (no optimizer step) on the host cores"},
        "cpu_baseline": {"value": val, "unit": "gates/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "gates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------- our arm (B200)
_SAVED_STDOUT = None


def _stdout_to_stderr():
    """Everything libraries write to file descriptor 1 while the benchmark runs (NCCL's version banner, the Trainer's
    device line) goes to stderr: stdout carries exactly ONE JSON line."""
    global _SAVED_STDOUT
    sys.stdout.flush()
    _SAVED_STDOUT = os.dup(1)
    os.dup2(2, 1)


def _restore_stdout():
    global _SAVED_STDOUT
    if _SAVED_STDOUT is not None:
        sys.stdout.flush()
        os.dup2(_SAVED_STDOUT, 1)
        os.close(_SAVED_STDOUT)
        _SAVED_STDOUT = None


def measure(w, wname, steps, warmup, nb, dev, rank, world, clocks_index=None, cpu_baseline=False, own_sizes=False,
            dump_dir=None):
    """Times `steps` train steps of workload `w` (after the setup pass and `warmup` steps) device-resident and end to end.
    Returns the record of this workload (the caller prints it, or nests it under "workloads").  `dump_dir`: where the
    outputs of the last step of the device-resident timed region (the one `value` comes from) are written."""
    import deepgate
    from deepgate import _native, ops
    from oracle import dg_oracle as O   # only for cpu_baseline (rank 0, N == 1) and the seeded weights helper
    variational = bool(w.get("variational", False))
    precision = w.get("precision", "fp32")
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, enable_reverse=True, s_rounds=4,
                                                     t_rounds=4, layernorm=True)
    mod = getattr(deepgate, "dg_ae_model_" + w["kind"])
    model = mod.Model(struct_encoder=enc, num_rounds=w["rounds"], dim_hidden=64, **({"variational": True} if variational else {}))
    sd = O.synth_state_dict(w["kind"], 2, variational=True) if variational else O.synth_state_dict(w["kind"], 2)
    model.load_state_dict(sd, strict=False)                # same random-init weights on every rank
    tmp = tempfile.mkdtemp(prefix="mgv_bench_")
    import contextlib
    # learning rate 0: the fused Adam kernel does all of its work (moments included) but leaves the weights at the seeded values,
    # so every step starts from the same weights in every run.  With a rate > 0 the weights drift apart between runs: the
    # backward's float atomics leave last-bit noise in the gradients, and Adam scales the gradients that are only noise (the
    # biases in front of the readout's BatchNorm: mathematically zero) up to full steps.
    with contextlib.redirect_stdout(sys.stderr):          # the Trainer prints its device like the reference's: stdout carries ONE JSON line
        trainer = deepgate.Trainer(None, model, training_id="bench", save_dir=tmp, lr=0.0,
                                   rc_prob_func_weight=list(LOSS_W), device=str(dev), batch_size=w["batch"],
                                   distributed=False)
    if variational:
        trainer.kl_weight = 1.0                            # cfg4: the KL term is part of the objective
    ops.set_precision(precision)
    model.train()
    host = [make_host_batch(w, rank, i, own_sizes).pack() for i in range(nb)]      # one pinned buffer per batch
    stats = [batch_stats(b, w["kind"]) for b in host]
    resident = [b.copy_to(dev, non_blocking=False) for b in host]
    gates_per_step = [s["gates"] * w["rounds"] for s in stats]

    def fresh(b):
        b._mgv_schedule = None            # a new batch every step: the level-CSR is rebuilt inside the step
        b.train_pos_edge_index = None
        return b

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize(dev)

    # only the step numbered keep["at"] holds on to its outputs: no step of a timed region runs with an earlier step's
    # outputs still allocated
    keep = {"at": -1}

    def step_resident(i):
        st = trainer.train_step(fresh(resident[i % nb]))
        if i == keep["at"]:
            keep["status"] = st
        return st["loss"]

    e2e_trace = [] if os.environ.get("MGV_BENCH_VERBOSE") else None

    class HostFeed(object):
        """The host batches in rotation, forever (what a DataLoader over pinned memory yields)."""
        def __iter__(self):
            i = 0
            while True:
                yield host[i % nb]
                i += 1

    # the package's own loader-side API: every step's batch is copied host -> device from pinned memory (one copy per step, issued on a
    # side stream while the previous step computes: deepgate.CudaPrefetcher, as Trainer.train does)
    feed = iter(deepgate.CudaPrefetcher(HostFeed(), dev, pin=False))

    # device -> host read of every step's result through the package's DeferredScalars (as Trainer.train does): the 4-byte copy
    # is issued behind the step, the host takes the value two steps later, and the values still in flight are read before the
    # closing event of the timed region (e2e_finish) -- every step's loss is read inside the region, none of the reads
    # empties the queue.  MGV_E2E_BLOCKING_READ=1 restores loss.item() inside the step (the reference's loop).
    blocking_read = bool(os.environ.get("MGV_E2E_BLOCKING_READ"))
    reader = deepgate.DeferredScalars(dev, lag=2)
    e2e_losses = []

    def step_e2e(i):
        t0 = time.perf_counter()
        b = next(feed)
        t1 = time.perf_counter()
        st = trainer.train_step(b)
        t2 = time.perf_counter()
        if blocking_read:
            e2e_losses.append(float(st["loss"].item()))
        else:
            done = reader.push(st["loss"])
            if done is not None:
                e2e_losses.append(done[0])
        if e2e_trace is not None:
            e2e_trace.append((1e3 * (t1 - t0), 1e3 * (t2 - t1), 1e3 * (time.perf_counter() - t2)))

    def e2e_finish():
        e2e_losses.extend(v[0] for v in reader.drain())

    def timed(fn, k, finish=None):
        import gc
        gc.collect()                    # no cyclic-GC pause (tens of ms) inside a timed region of a few steps
        gc.disable()
        try:
            return timed_(fn, k, finish)
        finally:
            gc.enable()

    def timed_(fn, k, finish):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(k):
            fn(i)
        if finish is not None:
            finish()
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=dev)
        if os.environ.get("MGV_BENCH_VERBOSE"):
            print("rank %d: %s: %d steps, %.2f ms on the device clock" % (rank, fn.__name__, k, float(ms.item())), file=sys.stderr)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return float(ms.item())

    sampler = ClockSampler(clocks_index) if clocks_index is not None else None
    if sampler:
        sampler.start()
    # setup (not a warm-up step): one pass over every DISTINCT batch so that the caching allocator owns blocks for
    # each batch's sizes -- a first-seen batch inside the timed region costs cudaMalloc calls of several hundred MB
    # (measured: 7.8 instead of 4.6 ms / step with --warmup 3 and 4 distinct batches)
    for i in range(nb):
        step_resident(i)
        step_e2e(i)
    for i in range(warmup):
        step_resident(i)
        step_e2e(i)
    # untimed: three rotations in the mode that is timed next -- the caching allocator re-settles when the step mix changes and a
    # cudaMalloc inside a timed step stalls it for 5-90 ms (max over ranks: one rank is enough)
    for i in range(max(3 * nb, 12)):
        step_resident(i)
    launches0 = _native.lib().mgv_kernel_launches()
    if sampler:
        sampler.mark_begin()
    mallocs0 = torch.cuda.memory_stats(dev).get("num_device_alloc", 0)
    keep["at"] = steps - 1 if dump_dir is not None else -1
    ms = timed(step_resident, steps)
    keep["at"] = -1
    mallocs_resident = torch.cuda.memory_stats(dev).get("num_device_alloc", 0) - mallocs0
    launches = _native.lib().mgv_kernel_launches() - launches0
    # copied to pageable host memory (no device allocation) before the next region; written after the last one
    outputs = {k: v.detach().cpu() for k, v in keep.pop("status", {}).items() if torch.is_tensor(v)}
    # the same K steps once more with a CUDA-event pair around every library call (the per-kernel table and the roofline's launch
    # durations): ~30 event pairs per step cost the host ~0.1 ms, so they stay out of the region `value` is taken from; the
    # profiled region's own time is reported next to it (`profiled_ms_per_step`)
    ops.PROFILE = {}
    ms_profiled = timed(step_resident, steps)
    if sampler:
        sampler.mark_end()
    torch.cuda.synchronize(dev)
    prof = ops.profile_summary()
    ops.PROFILE = None
    # clocks are sampled over the device-resident timed region only: nvidia-smi polling takes driver locks that the per-step
    # synchronising end-to-end loop is sensitive to
    clocks = sampler.stop() if sampler else None
    # untimed: back from the resident loop to the host-fed path, three rotations over the distinct batches.  The caching allocator
    # re-settles when the per-step batch copies join the working set: it issues one more cudaMalloc around the 11th host-fed step
    # (measured, deterministic), and that call stalls the step for 5-90 ms -- it must not land in the timed region.
    for i in range(max(3 * nb, 12)):
        step_e2e(i)
    alloc0 = torch.cuda.memory_stats(dev).get("num_device_alloc", 0)
    e2e_finish()
    del e2e_losses[:]
    ms_e2e = timed(step_e2e, steps, e2e_finish)
    if len(e2e_losses) != steps or not all(math.isfinite(v) for v in e2e_losses):
        raise RuntimeError("bench: the end-to-end region read %d finite losses for %d steps" % (len(e2e_losses), steps))
    mallocs_e2e = torch.cuda.memory_stats(dev).get("num_device_alloc", 0) - alloc0
    if os.environ.get("MGV_BENCH_VERBOSE"):
        print("cudaMalloc calls inside the timed regions: resident %d, end-to-end %d" % (mallocs_resident, mallocs_e2e), file=sys.stderr)
    if e2e_trace:
        for t in e2e_trace[-steps:]:
            print("e2e step: h2d issue %.2f  train_step host %.2f  loss read %.2f ms" % t, file=sys.stderr)
    from deepgate.schedule import check_deferred_errors
    check_deferred_errors()                   # asynchronous input validation of every schedule built above
    ops.set_precision("fp32")
    if dump_dir is not None:
        write_outputs(dump_dir, outputs)

    g_local = sum(gates_per_step[i % nb] for i in range(steps))
    g_all = torch.tensor([float(g_local)], device=dev, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(g_all)
    value = float(g_all.item()) / (ms * 1e-3)
    e2e = float(g_all.item()) / (ms_e2e * 1e-3)

    # ---- roofline of the dominant kernel (largest share of the timed region), algorithmic bytes per launch
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_source = "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650"
    tc_sweep = w["rounds"] == 1               # single-round sweeps run on the tcgen05 kernels (csrc/sweep_tc.cu)
    k_fwd, k_bwd = ("sweep_fwd_tc_kernel", "sweep_bwd_tc_kernel") if tc_sweep else ("sweep_fwd_kernel", "sweep_bwd_kernel")
    per_launch = {
        "level_sweep_fwd": (k_fwd, 1, "sweep_fwd_bytes"),
        "level_sweep_bwd": (k_bwd, 1, "sweep_bwd_bytes"),
        "struct_encoder_fwd": ("struct_fwd_tc_kernel", 8, "struct_fwd_bytes"),   # 2 * s_rounds step launches per call
        # backward step = struct_bwd_pw_kernel (recompute + pointwise + data gradient) followed by struct_bwd_wgrad_kernel
        # (weight gradient); the two are timed together (one library call) and share the step's algorithmic bytes
        "struct_encoder_bwd": ("struct_bwd_pw_kernel+struct_bwd_wgrad_kernel", 8, "struct_bwd_bytes"),
    }
    mean_stats = {k: sum(s[k] for s in stats) / len(stats) for k in stats[0]}
    kernels = {}
    for name, (kern, nl, key) in per_launch.items():
        if name in prof and prof[name][0] > 0:
            calls, tot = prof[name]
            avg_launch_ms = tot / calls / nl
            ach = mean_stats[key] * (w["rounds"] if "sweep" in name else 1) / (avg_launch_ms * 1e-3) / 1e9
            kernels[kern] = {"ms_per_step": tot / steps, "avg_launch_ms": avg_launch_ms, "launches_per_step": nl,
                             "achieved_gbs": ach, "frac": ach / peak}
    # every other library call that is bracketed by events (one or two launches each): ms per step
    other = {name: tot / steps for name, (calls, tot) in prof.items() if name not in per_launch and calls > 0}
    traffic_table = {}
    try:
        traffic_table = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json"))).get(wname, {})
    except Exception:
        pass

    def traffic_of(*kerns):
        """DRAM bytes per launch from the committed ncu --set full captures of this workload (else None)."""
        joined = traffic_table.get("+".join(kerns))
        if joined:
            return joined["dram_read_bytes"] + joined["dram_write_bytes"]
        tot = 0
        for k in kerns:
            ent = traffic_table.get(k)
            if not ent:
                return None
            tot += ent["dram_read_bytes"] + ent["dram_write_bytes"]
        return tot

    top = max(kernels, key=lambda k: kernels[k]["ms_per_step"]) if kernels else None
    roofline = None
    if top:
        roofline = {"kernel": top, "bound": "hbm", "achieved": kernels[top]["achieved_gbs"], "peak": peak,
                    "unit": "GB/s", "frac": kernels[top]["frac"], "traffic": traffic_of(*top.split("+")),
                    "algorithmic_bytes_per_launch": mean_stats[per_launch[[k for k, v in per_launch.items() if v[0] == top][0]][2]],
                    "peak_source": peak_source, "share_of_step": kernels[top]["ms_per_step"] / (ms_profiled / steps)}
    sweep_ms = sum(kernels[k]["ms_per_step"] for k in (k_fwd, k_bwd) if k in kernels)
    sweep = None
    if sweep_ms > 0:
        sweep_bytes = (mean_stats["sweep_fwd_bytes"] + mean_stats["sweep_bwd_bytes"]) * w["rounds"]
        ach = sweep_bytes / (sweep_ms * 1e-3) / 1e9
        sweep = {"gates_per_s": mean_stats["gates"] * w["rounds"] / (sweep_ms * 1e-3), "ms_fwd_bwd": sweep_ms,
                 "achieved_gbs": ach, "frac": ach / peak,
                 # the level-propagation kernels (forward + backward launch of a step) against the HBM roofline
                 "roofline": {"kernel": k_fwd + "+" + k_bwd, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                              "frac": ach / peak, "traffic": traffic_of(k_fwd, k_bwd),
                              "algorithmic_bytes_per_launch": sweep_bytes, "peak_source": peak_source,
                              "share_of_step": sweep_ms / (ms_profiled / steps)}}

    cpu = None
    if cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        P = cpu_params(w["kind"])
        ns = pick_sample(w)
        cpu_step(w["kind"], P, host[0], w["rounds"], max(1, ns // 4))        # warm-up
        dt, gates = cpu_step(w["kind"], P, host[0], w["rounds"], ns)
        cpu = {"value": gates / dt, "unit": "gates/s", "cores": cores, "kind": "port",
               "sample": "1 train step on %d of %d circuits (%d gates, %.1f s), oracle port with the reference's "
                         "per-node subgraph loop" % (ns, w["batch"], gates, dt)}
    h2d = sum(b.nbytes() for b in host) / len(host)
    losses = "recon/prob/func" + ("/KL" if variational else "")
    rec = {
        "metric": "gates_per_s_fwd_bwd", "value": value, "unit": "gates/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms / steps, "profiled_ms_per_step": ms_profiled / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": wname, "model": ("DG_VAE-" if variational else "DG_AE-") + w["kind"], "circuits_per_gpu": w["batch"],
                   "nodes_per_gpu": mean_stats["N"], "edges_per_gpu": mean_stats["E"], "levels": mean_stats["L"],
                   "gates_per_step_per_gpu": mean_stats["gates"] * w["rounds"], "sweep_rounds": w["rounds"],
                   "s_rounds": 4, "t_rounds": 4, "layernorm": True, "dim_hidden": 64, "parallelism": "dp%d" % world,
                   "step": "schedule build + forward + %s losses + backward + allreduce + Adam" % losses,
                   "ranks": ("every rank draws its own circuits AND its own circuit sizes (plain DistributedSampler)" if own_sizes else
                             "every rank draws its own circuits, with the same circuit sizes on all ranks (size-bucketed sampler)"),
                   "setup": "one untimed pass over each distinct batch before the warm-up steps (allocator pools)",
                   "e2e_feed": "deepgate.CudaPrefetcher over pinned host batches: one host->device copy per step, issued on a side stream "
                               "while the previous step computes (as Trainer.train does); every step's loss read back (e2e.result_read)",
                   "l2": "%d distinct batches rotated; per-batch working set (struct states %d MB) exceeds the 126 MB L2"
                         % (nb, int(2 * 9 * mean_stats["N"] * 256 / 1e6))},
        "e2e": {"value": e2e, "unit": "gates/s", "ms_per_step": ms_e2e / steps,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                "result_read": "loss.item() inside the step" if blocking_read else
                               "every step's loss copied to pinned host memory behind the step and read two steps later (deepgate.DeferredScalars, lag 2); all reads inside the timed region"},
        "gpu_launches": int(launches), "cuda_mallocs_in_timed_regions": {"resident": int(mallocs_resident), "e2e": int(mallocs_e2e)},
        "clocks": clocks, "roofline": roofline, "kernels": kernels, "other_calls_ms_per_step": other,
        "level_sweep": sweep, "cpu_baseline": cpu}
    # free this workload's device memory before the next one is measured
    del feed, trainer, model, resident, host
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return rec


# Workloads measured after the headline one and nested under "workloads" in the same JSON line (short runs: the named sizes
# of BASELINE.json's configs 3, 4 and 5 next to the headline config 2).
SUB_WORKLOADS = (("cfg5-k64", 3, 3, 1), ("cfg3-xmg", 5, 3, 2), ("cfg4", 5, 3, 2))      # name, steps, warm-up, distinct batches


def run_ours(args, w):
    _stdout_to_stderr()
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    # the step's random draws (edge order, negative samples, dropout masks) are seeded from torch's seed: fixed, so that the same
    # arguments give the same inputs in every run
    torch.manual_seed(rank)
    # clocks are sampled by rank 0 only (its GPU): one nvidia-smi poller per rank makes 8 processes hammer the driver's locks and
    # the host cores during the timed region of an 8-rank run
    rec = measure(w, args.workload, args.steps, args.warmup, args.batches, dev, rank, world, clocks_index=local if rank == 0 else None,
                  cpu_baseline=(rank == 0 and world == 1 and not args.no_cpu_baseline),
                  dump_dir=args.dump_outputs if rank == 0 else None)
    subs = {}
    if not args.no_sub_workloads and args.workload == "cfg2":
        for name, st, wu, nb in SUB_WORKLOADS:
            try:
                r = measure(WORKLOADS[name], name, st, wu, nb, dev, rank, world)
                subs[name] = {k: r[k] for k in ("value", "unit", "steps", "warmup", "ms_per_step", "dtype", "config", "e2e",
                                                 "gpu_launches", "roofline", "kernels", "level_sweep")}
            except Exception as e:                          # a sub-workload must never cost the headline line
                subs[name] = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
    rec["workloads"] = subs
    if world > 1 and not args.no_sub_workloads:
        # the same workload without the size-bucketed sampler: per-rank batches differ in nodes / levels, the step waits for the slowest rank
        try:
            r = measure(w, args.workload, min(args.steps, 10), 3, args.batches, dev, rank, world, own_sizes=True)
            rec["unbucketed_sizes"] = {k: r[k] for k in ("value", "unit", "steps", "warmup", "ms_per_step", "e2e", "config")}
        except Exception as e:
            rec["unbucketed_sizes"] = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
    if rank == 0:
        _restore_stdout()
        print(json.dumps(rec))
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--batches", type=int, default=4, help="distinct synthetic batches rotated through the steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub-workloads", action="store_true", help="skip the short cfg3 / cfg4 / cfg5 runs nested under 'workloads'")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl ours)")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
