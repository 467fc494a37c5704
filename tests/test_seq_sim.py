"""Sequential simulation of netlists with latches (simulate_counts / label_circuits with ``cycles``, csrc/logic_sim.cu's
seq_sim_kernel) against the numpy reference tests/seq_sim_oracle.py.
CPU: the reference's two identities with combinational simulation and its exact counts on a one-hot ring, a toggle
flip-flop, a 3-bit counter and a shift register; read_aiger's ``latches`` in both formats and its reset errors; argument
errors.  GPU: counts bit-equal to the reference for the four kinds on fixtures, random sequential AIGs, deep circuits,
partial slices, warm-up and the 200 k-AND netlist; the identities against simulate_counts itself; pass split and batch
independence; every latch validation error; mapping keeps sequential counts; the CLI through NpzParser and training."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import seq_sim_oracle as SQ
import test_aiger as TA
from oracle import logic_sim as OL

KINDS = ["aig", "mig", "xmg", "xag"]


class Seq(object):
    """Builds an ASCII AIGER file with latches, gate by gate, without simplifying."""

    def __init__(self):
        self.m, self.inputs, self.latches, self.ands, self.outputs = 0, [], [], [], []

    def var(self):
        self.m += 1
        return 2 * self.m

    def input(self):
        self.inputs.append(self.var())
        return self.inputs[-1]

    def latch(self, reset=0):
        """reset 0, 1 or "u" (uninitialised); the next state is set with ``next``."""
        v = self.var()
        self.latches.append([v, 0, v if reset == "u" else reset])
        return v

    def next(self, q, lit):
        [l for l in self.latches if l[0] == q][0][1] = lit

    def AND(self, a, b):
        v = self.var()
        self.ands.append((v, a, b))
        return v

    def XOR(self, a, b):
        return self.AND(self.AND(a, b ^ 1) ^ 1, self.AND(a ^ 1, b) ^ 1) ^ 1

    def text(self):
        rows = ["aag %d %d %d %d %d" % (self.m, len(self.inputs), len(self.latches), len(self.outputs), len(self.ands))]
        rows += ["%d" % i for i in self.inputs]
        rows += ["%d %d" % (q, n) if r == 0 else "%d %d %d" % (q, n, r) for q, n, r in self.latches]
        rows += ["%d" % o for o in self.outputs] + ["%d %d %d" % a for a in self.ands]
        return "\n".join(rows) + "\n"


def ring(k):
    """One-hot ring of k latches (latch 0 resets to 1), one primary input and the outputs AND(latch i, input)."""
    g = Seq()
    x = g.input()
    q = [g.latch(1 if i == 0 else 0) for i in range(k)]
    for i in range(k):
        g.next(q[i], q[i - 1])
    g.outputs += [g.AND(v, x) for v in q]
    return g.text()


def toggle():
    g = Seq()
    q = g.latch(0)
    g.next(q, q ^ 1)
    g.outputs.append(q)
    return g.text()


def counter3():
    """3-bit counter b2 b1 b0 with enable constant 1: bit i in cycle t is bit i of t mod 8."""
    g = Seq()
    b = [g.latch(0) for _ in range(3)]
    carry = 1
    for q in b:
        g.next(q, g.XOR(q, carry))
        carry = g.AND(q, carry)
    g.outputs.append(carry)
    return g.text()


def shift(n):
    """Shift register of n stages (all reset 1) fed by the primary input."""
    g = Seq()
    x = g.input()
    s = [g.latch(1) for _ in range(n)]
    for i in range(n):
        g.next(s[i], x if i == 0 else s[i - 1])
    g.outputs.append(s[-1])
    return g.text()


def random_seq(rng, I, L, A, resets=(0, 1, "u")):
    """A random sequential AIG: ANDs over any earlier variable (constants and repeats included, so folding happens);
    next states among constants, the latch itself, other latches and any literal; resets drawn from ``resets``."""
    g = Seq()
    for _ in range(I):
        g.input()
    q = [g.latch(resets[rng.integers(len(resets))]) for _ in range(L)]
    for _ in range(A):
        hi = g.m + 1
        g.AND(*(2 * int(rng.integers(0 if rng.random() < 0.05 else 1, hi)) + int(rng.integers(2)) for _ in range(2)))
    lits = 2 * (1 + np.arange(g.m)) if g.m else np.zeros(1, np.int64)
    for i, v in enumerate(q):
        kind = rng.integers(4)
        lit = [int(rng.integers(2)), v, q[rng.integers(L)], int(rng.choice(lits))][kind]
        g.next(v, lit ^ int(rng.integers(2)))
    g.outputs += [int(a[0]) ^ int(rng.integers(2)) for a in g.ands[-3:]]
    return g.text()


def read_text(tmp_path, name, text, kind="aig"):
    from deepgate.aiger import read_aiger
    return read_aiger(TA.write(tmp_path, name, text), kind)


def arrays(circuits):
    """(code, edge_index [2, E], batch, latches) of circuit dicts placed one after another."""
    from deepgate.simulate import _batch_latches
    n = np.cumsum([0] + [len(c["x"]) for c in circuits])
    code = np.concatenate([c["x"][:, 1] for c in circuits]).astype(np.int64)
    ei = np.concatenate([c["edge_index"].reshape(-1, 2) + n[i] for i, c in enumerate(circuits)]).T
    batch = np.repeat(np.arange(len(circuits)), np.diff(n))
    return code, ei, batch, _batch_latches(circuits).numpy()


def reference(circuits, kind, **kw):
    code, ei, batch, lat = arrays(circuits)
    return SQ.simulate(code, ei, kind, latches=lat, batch=batch, **kw)


# ------------------------------------------------------------------ reference (CPU)
def test_reference_without_latches_is_combinational_at_patterns_times_cycles():
    from deepgate import synth
    circuits = synth.make_circuits("xmg", 4, (8, 16), (60, 200), cfg=91, window=12, n_pairs=10)
    code, ei, batch, _ = arrays(circuits)
    pairs = np.random.default_rng(0).integers(0, len(code), (2, 30))
    got = SQ.simulate(code, ei, "xmg", batch=batch, pairs=pairs, patterns=128, seed=5, cycles=3)
    want = OL.simulate(code, ei, "xmg", batch=batch, pairs=pairs, patterns=384, seed=5)
    assert got[2] == want[2] and np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_reference_one_cycle_from_uninitialised_latches_is_combinational(tmp_path):
    rng = np.random.default_rng(1)
    circuits = [read_text(tmp_path, "r%d.aag" % i, random_seq(rng, 3, 4, 30, resets=("u",))) for i in range(8)]
    code, ei, batch, lat = arrays(circuits)
    got = SQ.simulate(code, ei, "aig", latches=lat, batch=batch, patterns=192, seed=3, cycles=1)
    want = OL.simulate(code, ei, "aig", batch=batch, patterns=192, seed=3)
    assert got[2] == want[2] and np.array_equal(got[0], want[0])


@pytest.mark.parametrize("k,cycles,warmup", [(3, 9, 0), (4, 12, 4), (5, 7, 2)])
def test_reference_one_hot_ring(tmp_path, k, cycles, warmup):
    c = read_text(tmp_path, "ring.aag", ring(k))
    ones, _, samples = reference([c], "aig", patterns=256, cycles=cycles, warmup=warmup)
    q = c["latches"][:, 0]
    assert list(q) == list(range(1, k + 1))
    want = [256 * sum((t - i) % k == 0 for t in range(warmup, cycles)) for i in range(k)]
    assert list(ones[q]) == want and samples == 256 * (cycles - warmup)
    if (cycles - warmup) % k == 0:
        assert all(ones[q] == samples // k)


def test_reference_toggle_flip_flop(tmp_path):
    c = read_text(tmp_path, "t.aag", toggle())
    ones, _, samples = reference([c], "aig", patterns=128, cycles=7, warmup=2)
    assert ones[c["latches"][0, 0]] == 128 * 2 and samples == 128 * 5          # odd t in [2, 7): 3, 5


def test_reference_three_bit_counter(tmp_path):
    c = read_text(tmp_path, "cnt.aag", counter3())
    cycles, warmup = 21, 3
    ones, _, _ = reference([c], "aig", patterns=64, cycles=cycles, warmup=warmup)
    for i, v in enumerate(c["latches"][:, 0]):
        assert ones[v] == 64 * sum((t >> i) & 1 for t in range(warmup, cycles)), i


def test_reference_shift_register(tmp_path):
    c = read_text(tmp_path, "sh.aag", shift(4))
    patterns, cycles, seed = 192, 6, 7
    T = patterns // 64
    ones, _, _ = reference([c], "aig", patterns=patterns, cycles=cycles, seed=seed)
    x = [OL.popcount(OL.input_words([0], u * T + np.arange(T), seed, False)).sum() for u in range(cycles)]
    for i, v in enumerate(c["latches"][:, 0]):           # stage i: its reset 1 while t <= i, then x of cycle t - 1 - i
        assert ones[v] == sum(patterns if t <= i else x[t - 1 - i] for t in range(cycles)), i


def test_reference_counts_do_not_depend_on_passes(tmp_path):
    rng = np.random.default_rng(2)
    circuits = [read_text(tmp_path, "r%d.aag" % i, random_seq(rng, 2, 3, 25)) for i in range(5)]
    code, ei, batch, lat = arrays(circuits)
    pairs = rng.integers(0, len(code), (2, 20))
    kw = dict(latches=lat, batch=batch, pairs=pairs, patterns=640, cycles=4, warmup=1)
    a, b = SQ.simulate(code, ei, "aig", **kw), SQ.simulate(code, ei, "aig", words_per_pass=3, **kw)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ------------------------------------------------------------------ read_aiger's latches (CPU)
def test_read_aiger_latches_in_both_formats(tmp_path):
    from deepgate.aiger import read_aiger
    text = "aag 6 1 4 1 1\n2\n4 12 0\n6 5\n8 3 1\n10 10 10\n12\n12 4 6\n"   # resets 0, none (0), 1, uninitialised
    a = read_text(tmp_path, "l.aag", text)
    data, _ = TA.to_binary(text)
    b = read_aiger(TA.write(tmp_path, "l.aig", data))
    assert np.array_equal(a["latches"], b["latches"])
    lat = a["latches"]
    assert lat.dtype == np.int64 and lat.shape == (4, 3)
    assert list(lat[:, 0]) == [1, 2, 3, 4] and list(lat[:, 2]) == [0, 0, 1, 2]
    assert np.array_equal(lat[:, 1], a["outputs"][1:5])
    assert read_text(tmp_path, "c.aag", TA.FIXTURES["consts"])["latches"].shape == (0, 3)
    for name in TA.FIXTURES:                                   # the existing fixtures' ASCII and binary twins agree
        data, _ = TA.to_binary(TA.FIXTURES[name])
        assert np.array_equal(read_text(tmp_path, name + ".aag", TA.FIXTURES[name])["latches"],
                              read_aiger(TA.write(tmp_path, name + ".aig", data))["latches"])


@pytest.mark.parametrize("reset", [2, 4, 9])
def test_invalid_reset_names_the_file_and_line(tmp_path, reset):
    import re
    from deepgate.aiger import read_aiger
    text = "aag 3 1 2 1 0\n2\n4 2\n6 4 %d\n4\n" % reset
    path = TA.write(tmp_path, "r.aag", text)
    with pytest.raises(ValueError, match="^" + re.escape(path) + ": line 4: latch reset %d must be 0, 1 or the latch "
                                         "literal 6" % reset):
        read_aiger(path)
    path = TA.write(tmp_path, "r.aig", TA.encode_binary(1, [2, 4], [0, reset], [4], (0, 0), np.zeros((0, 2), np.int64)))
    with pytest.raises(ValueError, match="^" + re.escape(path) + ": line 3: latch reset %d must be" % reset):
        read_aiger(path)


# ------------------------------------------------------------------ argument errors (CPU)
def test_cli_sequential_arguments(tmp_path):
    from deepgate.simulate import main
    a = TA.write(tmp_path, "ring.aag", ring(3))
    out = ["--out", str(tmp_path / "o")]
    for bad in (["--graphs", "g.npz", "--type", "mig", "--cycles", "4"],
                ["--aiger", a, "--type", "mig", "--cycles", "4", "--exhaustive"],
                ["--aiger", a, "--type", "mig", "--cycles", "4", "--class-pairs", "2"],
                ["--aiger", a, "--type", "mig", "--warmup", "2"],
                ["--aiger", a, "--type", "mig", "--cycles", "4", "--warmup", "4"],
                ["--aiger", a, "--type", "mig", "--cycles", "0"]):
        with pytest.raises(SystemExit):
            main(bad + out)


def test_api_sequential_argument_errors(tmp_path):
    import deepgate
    from deepgate.simulate import simulate_counts
    c = read_text(tmp_path, "ring.aag", ring(3))
    G = deepgate.circuits_to_batch([dict(c, prob=np.zeros(len(c["x"]), np.float32), tt_sim=np.zeros(0, np.float32),
                                         tt_pair_index=np.zeros((0, 2), np.int64))])
    lat = c["latches"]
    for kw, msg in ((dict(cycles=4, exhaustive=True), "exhaustive"), (dict(cycles=0), "cycles"),
                    (dict(cycles=2 ** 31), "cycles"), (dict(cycles=2 ** 27, patterns=2 ** 20), "cycles"), (dict(cycles=4, warmup=4), "warmup"),
                    (dict(cycles=4, warmup=-1), "warmup"), (dict(warmup=1), "need cycles"),
                    (dict(latches=lat), "need cycles"), (dict(cycles=4, latches=lat[:, :2]), r"\[L, 3\]")):
        kw.setdefault("latches", lat if "cycles" in kw else None)
        with pytest.raises(ValueError, match=msg):
            simulate_counts(G, "aig", **kw)
    with pytest.raises(ValueError, match="class_pairs"):
        deepgate.label_circuits([c], "aig", "cpu", class_pairs=4, cycles=4)
    with pytest.raises(ValueError, match="latches"):
        deepgate.label_circuits([c], "aig", "cpu", cycles=4, latches=lat)


# ------------------------------------------------------------------ GPU
def batch(circuits, n_pairs=12, seed=0):
    """CUDA batch of circuit dicts with random pairs, and their batch-global latches."""
    import deepgate
    from deepgate.simulate import _batch_latches
    rng = np.random.default_rng(seed)
    chunk = [{"x": c["x"], "edge_index": c["edge_index"], "prob": np.zeros(len(c["x"]), np.float32),
              "tt_sim": np.zeros(n_pairs, np.float32), "tt_pair_index": rng.integers(0, len(c["x"]), (n_pairs, 2))}
             for c in circuits]
    return deepgate.circuits_to_batch(chunk, "cuda"), _batch_latches(circuits)


def gpu(G, lat, kind, **kw):
    from deepgate.simulate import simulate_counts
    ones, diff, samples = simulate_counts(G, kind, latches=lat, **kw)
    return ones.cpu().numpy(), diff.cpu().numpy(), samples


def ref(G, lat, kind, **kw):
    return SQ.simulate(G.gate.reshape(-1).long().cpu().numpy(), G.edge_index.cpu().numpy(), kind, latches=lat.numpy(),
                       batch=G.batch.cpu().numpy(), pairs=G.tt_pair_index.cpu().numpy(), **kw)


def assert_same(got, want):
    assert got[2] == want[2]
    assert np.array_equal(got[0], want[0]), int(np.flatnonzero(got[0] != want[0])[0])
    assert np.array_equal(got[1], want[1])


def hand_and_random(tmp_path, kind, n_random=200, seed=11):
    texts = dict(TA.FIXTURES, ring3=ring(3), ring4=ring(4), toggle=toggle(), counter=counter3(), shift=shift(5))
    rng = np.random.default_rng(seed)
    for i in range(n_random):
        texts["r%03d" % i] = random_seq(rng, int(rng.integers(0, 6)), int(rng.integers(1, 8)), int(rng.integers(0, 60)))
    return [read_text(tmp_path, name + ".aag", t, kind) for name, t in sorted(texts.items())]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("warmup", [0, 3])
def test_counts_match_reference(tmp_path, kind, warmup):
    """Fixtures, hand circuits and 200 random sequential AIGs; 320 traces = 5 words: the second slice is partial."""
    G, lat = batch(hand_and_random(tmp_path, kind))
    kw = dict(patterns=320, seed=9, cycles=7, warmup=warmup)
    assert_same(gpu(G, lat, kind, **kw), ref(G, lat, kind, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_deep_circuit_matches_reference(tmp_path, kind):
    rng = np.random.default_rng(12)
    g = Seq()
    x = [g.input() for _ in range(4)]
    q = [g.latch(r) for r in (0, 1, "u", 0, 1, "u")]
    prev = x[0]
    for i in range(1300):                                    # a chain: AND i takes AND i - 1
        prev = g.AND(prev ^ int(rng.integers(2)), int(rng.choice(x + q)) ^ int(rng.integers(2)))
        if i % 250 == 100:
            g.next(q[i // 250], prev ^ 1)
    g.next(q[5], q[4])
    g.outputs.append(prev)
    c = read_text(tmp_path, "deep.aag", g.text(), kind)
    G, lat = batch([c])
    assert int(G.forward_level.max()) + 1 > 1000
    kw = dict(patterns=448, seed=1, cycles=5, warmup=1)
    assert_same(gpu(G, lat, kind, **kw), ref(G, lat, kind, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_200k_and_netlist_matches_reference(tmp_path, kind):
    from deepgate.aiger import read_aiger
    data, _ = TA.random_aig(64, 512, 200_000, 800, seed=3)
    c = read_aiger(TA.write(tmp_path, "seq200k.aig", data), kind)
    G, lat = batch([c], n_pairs=64)
    assert lat.shape == (512, 3)
    kw = dict(patterns=4096, seed=2, cycles=3, warmup=1)
    assert_same(gpu(G, lat, kind, **kw), ref(G, lat, kind, **kw))


@pytest.mark.gpu
def test_identities_against_combinational_simulate_counts(tmp_path):
    from deepgate import synth
    from deepgate.simulate import simulate_counts
    G, _ = batch(synth.make_circuits("mig4", 8, (8, 24), (100, 400), cfg=92, window=20))
    a = gpu(G, None, "mig", patterns=256, seed=4, cycles=5)
    b = simulate_counts(G, "mig", patterns=1280, seed=4)
    assert a[2] == b[2] and np.array_equal(a[0], b[0].cpu().numpy()) and np.array_equal(a[1], b[1].cpu().numpy())
    rng = np.random.default_rng(3)
    G, lat = batch([read_text(tmp_path, "u%d.aag" % i, random_seq(rng, 3, 5, 40, resets=("u",)), "xag")
                    for i in range(10)])
    a = gpu(G, lat, "xag", patterns=320, seed=6, cycles=1)
    b = simulate_counts(G, "xag", patterns=320, seed=6)
    assert a[2] == b[2] and np.array_equal(a[0], b[0].cpu().numpy()) and np.array_equal(a[1], b[1].cpu().numpy())


@pytest.mark.gpu
def test_counts_do_not_depend_on_passes_or_batch(tmp_path):
    import deepgate
    rng = np.random.default_rng(4)
    circuits = [read_text(tmp_path, "r%d.aag" % i, random_seq(rng, 4, 6, 80), "xmg") for i in range(16)]
    G, lat = batch(circuits)
    n = G.x.size(0)
    kw = dict(patterns=2048, seed=8, cycles=6, warmup=2)
    one = gpu(G, lat, "xmg", **kw)
    per = 8 * (n + len(lat))                                 # bytes per word of a pass (simulate._Sim.words_per_pass)
    split = gpu(G, lat, "xmg", max_bytes=4 * n + 8 * per, **kw)          # 8 of 32 words per pass: 4 passes
    assert_same(split, one)
    G9, lat9 = batch(circuits[9:10])
    alone = deepgate.simulate(G9, "xmg", latches=lat9, **kw)[0]
    prob = deepgate.simulate(G, "xmg", latches=lat, **kw)[0]
    s = sum(len(c["x"]) for c in circuits[:9])
    assert torch.equal(alone, prob[s:s + len(circuits[9]["x"])])


def latch_error(case, n, gate, other):
    """Row of latch 1 and the message for a batch of n nodes whose circuit 0 has INPUTs 0 .. 4 and a gate node ``gate``,
    and whose circuit 1 holds node ``other``."""
    return [([n + 5, 0, 0], "latch 1: node %d is outside \\[0, %d\\)" % (n + 5, n)),
            ([gate, 0, 0], "latch 1: node %d is not an INPUT" % gate),
            ([0, 0, 0], "latch 1: node 0 appears twice \\(also latch 0\\)"),
            ([1, 2 * n + 6, 0], "latch 1: next-state literal %d names a node outside" % (2 * n + 6)),
            ([1, -3, 0], "latch 1: next-state literal -3 names a node outside"),
            ([1, 2 * other + 1, 0], "latch 1: next-state literal %d names a node of another circuit" % (2 * other + 1)),
            ([1, 0, 3], "latch 1: reset 3 is not 0, 1 or 2")][case]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(7))
def test_latch_validation_names_the_latch(tmp_path, case):
    from deepgate.simulate import simulate_counts
    rng = np.random.default_rng(5)
    a = read_text(tmp_path, "a.aag", random_seq(rng, 2, 3, 20))
    G, _ = batch([a, read_text(tmp_path, "b.aag", random_seq(rng, 2, 3, 20))])
    n = G.x.size(0)
    lat = np.array([[0, 0, 0], [1, 0, 0], [2, 1, 2]], np.int64)
    row, msg = latch_error(case, n, int(np.flatnonzero(a["x"][:, 1] != 0)[0]), n - 1)
    lat[1] = row
    with pytest.raises(RuntimeError, match=msg):
        simulate_counts(G, "aig", patterns=128, cycles=3, latches=torch.from_numpy(lat))


@pytest.mark.gpu
def test_mapping_keeps_sequential_counts(tmp_path):
    from deepgate.aiger import read_aiger
    from deepgate.mapping import map_circuits
    data, _ = TA.random_aig(64, 512, 200_000, 800, seed=3)
    c = read_aiger(TA.write(tmp_path, "seq200k.aig", data), "aig")
    m = map_circuits([c], "xmg", "cuda:0")[0]
    assert np.array_equal(m["latches"][:, 0], c["latches"][:, 0]) and np.array_equal(m["latches"][:, 2],
                                                                                     c["latches"][:, 2])
    kw = dict(patterns=4096, seed=3, cycles=4, warmup=1)
    ones_a, _, samples = gpu(*batch([c], n_pairs=0), "aig", **kw)
    ones_m, _, _ = gpu(*batch([m], n_pairs=0), "xmg", **kw)
    o = m["origin"]
    want = np.where(o & 1, samples - ones_a[o >> 1], ones_a[o >> 1])
    assert (o & 1).any() and np.array_equal(ones_m, want)


@pytest.mark.gpu
def test_cli_sequential_to_training(tmp_path):
    import types
    import deepgate
    d = tmp_path / "netlists"
    d.mkdir()
    TA.write(d, "ring4.aag", ring(4))
    for i in range(3):
        TA.write(d, "small%d.aig" % i, TA.random_aig(8, 4, 300, 50, seed=4 + i, n_out=8)[0])
    TA.write(d, "adder.aag", TA.adder(4))
    out = tmp_path / "ds"
    env = dict(os.environ)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(root, "multi-gate-vae_b200"), env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, "-m", "deepgate.simulate", "--aiger", str(d), "--type", "xmg", "--map",
                        "--cycles", "32", "--warmup", "8", "--out", str(out)], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "simulating 16 latches over 32 cycles (24 counted)" in r.stdout and "labelled 5 circuits" in r.stdout
    labels = np.load(str(out / "labels.npz"), allow_pickle=True)["labels"].item()
    assert np.array_equal(labels["ring4"]["prob"][1:5], np.full(4, 0.25, np.float32))
    from deepgate.aiger import read_aiger
    from deepgate.mapping import map_circuits
    comb = deepgate.label_circuits(map_circuits([read_aiger(str(d / "ring4.aag"))], "xmg", "cuda:0"), "xmg", "cuda:0")
    assert np.all(np.abs(comb[0]["prob"][1:5] - 0.5) < 0.02)
    torch.manual_seed(0)
    parser = deepgate.NpzParser(str(out), str(out / "graphs.npz"), str(out / "labels.npz"), "xmg", random_shuffle=False,
                                trainval_split=0.6)
    train, val = parser.get_dataset()
    assert len(train) + len(val) == 5
    enc = deepgate.digae_layer.DirectMultiGCNEncoder(dim_hidden=64, dim_feature=6, s_rounds=1, t_rounds=1)
    model = deepgate.dg_ae_model_xmg.Model(struct_encoder=enc, dim_hidden=64)
    args = types.SimpleNamespace(model="DG_AE", type="xmg")
    trainer = deepgate.Trainer(args, model, training_id="seq", save_dir=str(tmp_path / "exp"), device="cuda:0",
                               batch_size=1, distributed=False, rc_prob_func_weight=[1.0, 4.0, 4.0])
    trainer.train(1, train, val)
    log = open(trainer.log_path).read()
    assert "train|" in log and "nan" not in log.lower()
