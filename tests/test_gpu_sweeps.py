"""The sweep kernels of klu_sweep.cu per state, at every instantiation and branch.

The log sweeps (`k_log_sweeps<G>`) stage the arcs of a batch of states in shared memory
(kCap arcs per tile), keep recent state scores in a ring (kRing slots) and switch on the
number of terms of a state (one or two: Kaldi's LogAdd; more: a streaming sum around a
shared reference point, redone exactly when it leaves [1e-280, 1e280]; more arcs than the
tile stages: the exact one-lane sum).  Every one of those switches moves with G.  The
builders below put states exactly at, below and above each switch for a given (G, kCap,
kRing) and every state's alpha and beta is compared with the oracle's
ComputeLatticeAlphasAndBetas restatement.

Also here: the tropical sweeps at each `pick_group` width (through lattice-prune-dyn-beam and
lattice-best-path2), the pieces of `k_banded_alpha` (through the position tools), and the
f64 `fast_exp` / `fast_log` / `log_add` of klu_common.cuh against long-double references."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from util import assert_rows_match

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "kaldi-lattice-utils_b200")

# ---- the constants of klu_sweep.cu, restated ---------------------------------------------------
# k_log_sweeps<G>:         kCap = kSweepCapPerLane * G = 8 G arcs per batch, kRing = sweep_ring(G)
# k_banded_alpha:          pieces of <= kBandStates = 128 states and <= kBandArcs = 768 arcs
# k_trop_sweeps<G>:        G = pick_group(arcs / states of the batch)
GROUPS = (2, 4, 8, 16, 32)
BAND_STATES, BAND_ARCS = 128, 768


def sweep_ring(g):
    return 128 if g >= 8 else 32


def sweep_consts(g):
    """(kCap, kRing) of the kernel run_log_sweeps launches at lane width g."""
    return 8 * g, sweep_ring(g)


def pick_group(avg_deg):
    if avg_deg <= 3.0:
        return 2
    if avg_deg <= 6.0:
        return 4
    if avg_deg <= 48.0:
        return 8
    if avg_deg <= 160.0:
        return 16
    return 32


FLAGS = [dict(), dict(acoustic_scale=0.1), dict(graph_scale=0.7, insertion_penalty=0.5)]
FLAG_IDS = ["plain", "ac0.1", "gs0.7+pen"]


# ---- lattices whose packed numbering is their input numbering ----------------------------------
def levels_of(nstates, arcs):
    """The packer's level: longest arc distance from any state without incoming arcs."""
    lvl = np.zeros(nstates, np.int64)
    for s, d, *_ in sorted(arcs, key=lambda a: a[0]):
        assert s < d, "builders number states in level order"
        lvl[d] = max(lvl[d], lvl[s] + 1)
    return lvl


def build(klu, key, nstates, arcs, finals, labels=None):
    """arcs: (src, dst, graph, acoustic[, label]).  States must be numbered by (level, id) --
    then the packed state ids the kernels see are these ids plus the lattice's offset, and
    the ring distances the builders aim at are the ones the kernel measures.  Durations are
    level differences, so the state times are consistent (the index tools accept it)."""
    lvl = levels_of(nstates, arcs)
    assert (np.diff(lvl) >= 0).all(), key + ": states are not in level order"
    full = []
    for i, a in enumerate(arcs):
        s, d, g, ac = a[:4]
        lab = a[4] if len(a) > 4 else 1 + (i % 7)
        full.append((s, d, lab, g, ac, int(lvl[d] - lvl[s])))
    return klu.make_lattice(key, nstates, full, finals)


def ring_lattice(klu, rng, g, cap, ring):
    """A chain P, one level W of g + 3 states (so at least two batches), a chain Q.  The
    first and last W state take arcs from P at exactly ring - 1, ring, ring + 1 and ring + 2
    states before W's end (forward: ring hit for <= ring, gather above) and send arcs to Q at
    exactly ring - 1, ring and ring + 1 states after W's start (backward)."""
    w = g + 3
    k = ring + 4
    a0, a1 = k, k + w
    n = a1 + k
    arcs = [(i, i + 1, *rng.uniform(0, 3, 2)) for i in range(k - 1)]
    arcs += [(i, i + 1, *rng.uniform(0, 3, 2)) for i in range(0, k - 1, 3)]  # parallel: 2-term states
    for s in range(a0, a1):
        arcs.append((k - 1, s, *rng.uniform(0, 3, 2)))
        arcs.append((s, a1, *rng.uniform(0, 3, 2)))
    for s in (a0, a1 - 1):
        for dist in (ring - 1, ring, ring + 1, ring + 2):
            arcs.append((a1 - dist, s, *rng.uniform(0, 3, 2)))
        for dist in (ring - 1, ring, ring + 1):
            arcs.append((s, a0 + dist, *rng.uniform(0, 3, 2)))
    arcs += [(i, i + 1, *rng.uniform(0, 3, 2)) for i in range(a1, n - 1)]
    finals = {n - 1: (0.5, 0.25), a0 + 1: (1.5, 0.5), a1 + 2: (2.0, 0.0)}
    return build(klu, "ring", n, arcs, finals)


def cap_lattice(klu, rng, cap, forward):
    """States whose arc count (in-arcs when `forward`, else out-arcs) is exactly cap - 1, cap
    and cap + 1, two of each in one level between small ones, and pairs that fill a batch to
    exactly cap arcs or one more.  The arcs run between a 12-state level and the probed level."""
    m = 12
    degs = [3]
    for d in (cap - 1, cap, cap + 1):
        degs += [d, 3, d, 3]
    degs += [cap // 2, cap - cap // 2, cap // 2, cap - cap // 2 + 1, 1, 1, 2]
    arcs, finals = [], {}
    if forward:
        # 0 -> sources 1..m -> probed states -> final
        src = list(range(1, m + 1))
        first = m + 1
        fin = first + len(degs)
        arcs += [(0, s, *rng.uniform(0, 2, 2)) for s in src]
        for i, d in enumerate(degs):
            arcs += [(src[(i + e) % m], first + i, *rng.uniform(0, 4, 2)) for e in range(d)]
            arcs.append((first + i, fin, *rng.uniform(0, 2, 2)))
        n = fin + 1
    else:
        # 0 -> probed states -> sinks -> final
        first = 1
        sinks = list(range(first + len(degs), first + len(degs) + m))
        fin = sinks[-1] + 1
        for i, d in enumerate(degs):
            arcs.append((0, first + i, *rng.uniform(0, 2, 2)))
            arcs += [(first + i, sinks[(i + e) % m], *rng.uniform(0, 4, 2)) for e in range(d)]
        arcs += [(s, fin, *rng.uniform(0, 2, 2)) for s in sinks]
        n = fin + 1
        finals[first + 1] = (1.0, 0.5)
    finals[n - 1] = (0.5, 0.5)
    return build(klu, "cap%s" % ("in" if forward else "out"), n, arcs, finals)


def level_sizes_lattice(klu, rng, g, ring):
    """Levels of 1, g - 1, g, g + 1, ring and ring + 1 states (and back to 1 between them):
    every state has two arcs from random states of the level below, one from its first state
    (so the levels are exact), and a third from two levels down now and then."""
    sizes = [1, 1, max(g - 1, 1), g, g + 1, 1, ring, ring + 1, 2, ring + 1, ring, 1, 1]
    starts = np.concatenate([[0], np.cumsum(sizes)])
    arcs = []
    for k in range(1, len(sizes)):
        prev = range(starts[k - 1], starts[k])
        for s in range(starts[k], starts[k + 1]):
            arcs.append((int(prev[0]), s, *rng.uniform(0, 3, 2)))
            arcs.append((int(rng.choice(prev)), s, *rng.uniform(0, 3, 2)))
            if k >= 2 and rng.rand() < 0.3:
                arcs.append((int(rng.randint(starts[k - 2], starts[k - 1])), s, *rng.uniform(0, 3, 2)))
    n = int(starts[-1])
    finals = {n - 1: (0.0, 0.5)}
    for s in rng.choice(n - 1, 5, replace=False):
        finals[int(s)] = (float(rng.uniform(2, 5)), 0.0)
    return build(klu, "levels", n, arcs, finals)


def narrow_wide_lattice(klu, rng, ring, forward):
    """A level of 2 states next to a level of ring + 8: one of the two has three arcs (a fast
    path sum) to / from the wide level's first and last states, the other covers the rest.
    Backward, the wide level's state t and t + ring share a ring slot and t + ring is written
    after t."""
    w = ring + 8
    if not forward:
        # 0 -> {A=1, B=2} -> W = 3 .. 3+w-1 -> F
        W = list(range(3, 3 + w))
        f = 3 + w
        arcs = [(0, 1, *rng.uniform(0, 2, 2)), (0, 2, *rng.uniform(0, 2, 2))]
        arcs += [(1, W[i], *rng.uniform(0, 3, 2)) for i in (0, 1, w - 1)]
        arcs += [(2, s, *rng.uniform(0, 3, 2)) for s in W]
        arcs += [(s, f, *rng.uniform(0, 6, 2)) for s in W]
        finals = {f: (0.0, 0.0), W[0]: (0.5, 0.5)}
        n = f + 1
    else:
        # 0 -> W = 1 .. w -> {A, B} -> F   (and the start's own beta reads the wide level)
        W = list(range(1, 1 + w))
        A, B, f = w + 1, w + 2, w + 3
        arcs = [(0, s, *rng.uniform(0, 6, 2)) for s in W]
        arcs += [(W[i], A, *rng.uniform(0, 3, 2)) for i in (0, w - 2, w - 1)]
        arcs += [(s, B, *rng.uniform(0, 3, 2)) for s in W]
        arcs += [(A, f, 1.0, 0.5), (B, f, 0.5, 1.0)]
        finals = {f: (0.0, 0.0)}
        n = f + 1
    return build(klu, "narrowwide", n, arcs, finals)


def terms_lattice(klu, rng):
    """States with 1, 2 and 3 terms in each direction, a final weight counting as one."""
    # 0 -> a (1 arc), b (2 parallel), c (3 parallel); a, b, c -> d ; finals on a (1 term back),
    # b (final + 1 arc), c (final + 2 arcs)
    arcs = [(0, 1, 1.0, 0.5), (0, 2, 0.3, 0.1), (0, 2, 0.7, 0.2), (0, 3, 0.2, 0.2), (0, 3, 1.2, 0.1),
            (0, 3, 0.9, 0.9), (2, 4, 0.5, 0.5), (3, 4, 0.25, 0.5), (3, 4, 1.5, 0.1), (4, 5, 0.1, 0.1)]
    finals = {1: (0.5, 0.0), 2: (1.0, 0.0), 3: (2.0, 1.0), 5: (0.0, 0.0)}
    return build(klu, "terms", 6, arcs, finals)


def range_lattice(klu, rng):
    """Dynamic range: arcs 600-2000 nats apart into one state; a state whose terms are ~700
    nats from the reference point (the previous batch's first state) on either side; states
    that nothing reaches (alpha -inf, also with three -inf terms) and dead ends (beta -inf)."""
    arcs = [
        # 0 start, 1 and 2 unreachable sources (level 0)
        (0, 3, 0.5, 0.5), (1, 3, 1.0, 1.0), (1, 4, 0.5, 0.5), (2, 4, 0.5, 0.5), (1, 4, 2.0, 0.0),
        # 3 -> 5 with terms 600, 1400 and 2000 nats above the best one
        (3, 5, 1.0, 0.0), (3, 5, 601.0, 0.0), (3, 5, 1001.0, 400.0), (3, 5, 1000.0, 1001.0),
        # 5 -> 6: three terms ~700 nats above the reference (alpha[5]), then 6 -> 7 back down
        (5, 6, -350.0, -350.0), (5, 6, -350.0, -350.5), (5, 6, -351.0, -350.0),
        (6, 7, 700.0, 0.5), (6, 7, 700.5, 0.0), (6, 7, 701.0, 0.25),
        # 7 -> 8 three terms 700 nats below
        (7, 8, 700.0, 0.0), (7, 8, 350.0, 351.0), (7, 8, 702.0, 0.0),
        # 4 (reached only from unreachable states) -> 8; 8 -> 9 (dead end) and 8 -> 10 (final)
        (4, 8, 0.5, 0.5), (8, 9, 0.5, 0.5), (8, 10, 0.1, 0.2), (8, 10, 0.3, 0.2), (8, 10, 0.5, 0.1),
    ]
    return build(klu, "range", 11, arcs, {10: (0.0, 0.0), 7: (900.0, 0.0)})


def diamond_lattice(klu, rng, n=40):
    """Chains of diamonds: every state has at most two terms in both directions."""
    arcs, s = [], 0
    for _ in range(n):
        arcs += [(s, s + 1, *rng.uniform(0, 3, 2)), (s, s + 2, *rng.uniform(0, 3, 2)),
                 (s + 1, s + 3, *rng.uniform(0, 3, 2)), (s + 2, s + 3, *rng.uniform(0, 3, 2))]
        s += 3
    return build(klu, "diamonds", s + 1, arcs, {s: (0.5, 0.5)})


def adversarial(klu, g, seed=0):
    cap, ring = sweep_consts(g)
    rng = np.random.RandomState(1000 + g + seed)
    return [ring_lattice(klu, rng, g, cap, ring), cap_lattice(klu, rng, cap, True), cap_lattice(klu, rng, cap, False),
            level_sizes_lattice(klu, rng, g, ring), narrow_wide_lattice(klu, rng, ring, True),
            narrow_wide_lattice(klu, rng, ring, False), terms_lattice(klu, rng), range_lattice(klu, rng),
            diamond_lattice(klu, rng)]


# ---- comparison with the oracle ---------------------------------------------------------------
def check_states(got, want, what):
    """-inf in the same places, every finite value within 1e-9 relative."""
    for name, g, w in zip(("alpha", "beta"), got[:2], want[:2]):
        assert np.array_equal(np.isneginf(g), np.isneginf(w)), "%s: %s -inf differs at %s" % (
            what, name, np.flatnonzero(np.isneginf(g) != np.isneginf(w))[:8])
        assert np.isfinite(w[~np.isneginf(w)]).all() and np.isfinite(g[~np.isneginf(g)]).all()
        fin = np.isfinite(w)
        if fin.any():
            err = np.abs(g[fin] - w[fin]) / np.maximum(1.0, np.abs(w[fin]))
            k = int(np.argmax(err))
            assert err[k] <= 1e-9, "%s: %s of state %d: %r vs %r" % (what, name, np.flatnonzero(fin)[k],
                                                                        g[fin][k], w[fin][k])
    gt, wt = got[2], want[2]
    assert (np.isinf(gt) and gt == wt) or abs(gt - wt) <= 1e-9 * max(1.0, abs(wt)), "%s: total %r vs %r" % (what, gt, wt)


def run_fwd_bwd(klu, engine, batch, **flags):
    engine.load(batch)
    engine.run(klu.FWD_BWD, **flags)
    return engine.fetch_fwd_bwd()


def check_batch(ora, batch, res, flags, what, only=None):
    al, be, tot = res
    for l in (range(len(batch)) if only is None else only):
        lat = batch[l]
        a, b = int(batch.state_off[l]), int(batch.state_off[l + 1])
        if b == a:
            assert tot[l] == 0.0
            continue
        check_states((al[a:b], be[a:b], tot[l]), ora.fwd_bwd(lat, **flags), "%s lattice %d (%s)" % (what, l, lat.key))


def ragged(klu):
    """Empty and one-state lattices between synthetic ones."""
    one = klu.make_lattice("one", 1, [], {0: (0.5, 0.5)})
    nofinal = klu.make_lattice("nofinal", 1, [], {})
    empty = klu.make_lattice("empty", 0, [], {})
    syn = klu.synth_batch("tiny", 4, seed=12).lattices()
    return [empty, syn[0], one, empty, syn[1], nofinal, syn[2], one, syn[3], empty]


# ---- 2. the log sweeps at every lane width -----------------------------------------------------
@pytest.mark.parametrize("flags", FLAGS, ids=FLAG_IDS)
@pytest.mark.parametrize("g", GROUPS)
def test_log_sweeps_adversarial(klu, ora, engine, monkeypatch, g, flags):
    """Every builder at lane width g (KLU_SWEEP_LANES, read on every run), per state."""
    monkeypatch.setenv("KLU_SWEEP_LANES", str(g))
    lats = adversarial(klu, g)
    batch = klu.LatticeBatch.from_lattices(lats)
    check_batch(ora, batch, run_fwd_bwd(klu, engine, batch, **flags), flags, "G=%d" % g)


@pytest.mark.parametrize("g", GROUPS)
def test_log_sweeps_synthetic_and_ragged(klu, ora, engine, monkeypatch, g):
    """tiny, small and c2 batches and a ragged one (empty and one-state lattices) at width g."""
    monkeypatch.setenv("KLU_SWEEP_LANES", str(g))
    lats = (klu.synth_batch("tiny", 10, seed=40 + g).lattices() + klu.synth_batch("small", 6, seed=50 + g).lattices() +
            klu.synth_batch("c2", 2, seed=60 + g).lattices() + ragged(klu))
    batch = klu.LatticeBatch.from_lattices(lats)
    for flags in FLAGS:
        check_batch(ora, batch, run_fwd_bwd(klu, engine, batch, **flags), flags, "G=%d %r" % (g, flags))


def _host_prune(lat, beam, flags):
    """PruneLattice's arc and final tests as the sweeps evaluate them (arc_pruned /
    final_pruned): tropical forward / backward costs in double with the same order of
    additions, the arc dropped when fwd[s] + (cost + bwd[d]) > best + beam.  Returns the
    lattice without the dropped arcs and finals (state ids unchanged)."""
    gs = np.float32(flags.get("graph_scale", 1.0))
    as_ = np.float32(flags.get("acoustic_scale", 1.0))
    pen = np.float32(flags.get("insertion_penalty", 0.0))
    scale = gs != 1 or as_ != 1

    def cost(g, a, lab):
        g, a = np.float32(g), np.float32(a)
        if scale and not (np.isposinf(g) and np.isposinf(a)):
            g, a = np.float32(gs * g), np.float32(as_ * a)
        if lab != 0:
            g = np.float32(g + pen)
        return float(np.float64(g) + np.float64(a))

    n = lat.nstates
    c = [cost(lat.graph[e], lat.acoustic[e], lat.label[e]) for e in range(lat.narcs)]
    fc = [cost(lat.fin_graph[s], lat.fin_acoustic[s], 0) for s in range(n)]
    fwd = [np.inf] * n
    fwd[0] = 0.0
    order = np.argsort(lat.dst, kind="stable")
    for e in order:
        s, d = int(lat.src[e]), int(lat.dst[e])
        fwd[d] = min(fwd[d], fwd[s] + c[e])
    bwd = list(fc)
    for e in np.argsort(-lat.src, kind="stable"):
        s, d = int(lat.src[e]), int(lat.dst[e])
        bwd[s] = min(bwd[s], c[e] + bwd[d])
    best = min(fwd[s] + fc[s] for s in range(n))
    lim = best + float(np.float32(beam))
    keep = [e for e in range(lat.narcs) if not (fwd[int(lat.src[e])] + (c[e] + bwd[int(lat.dst[e])]) > lim)]
    fin = {s: (float(lat.fin_graph[s]), float(lat.fin_acoustic[s])) for s in range(n)
           if np.isfinite(fc[s]) and not (fc[s] + fwd[s] > lim)}
    arcs = [(int(lat.src[e]), int(lat.dst[e]), int(lat.label[e]), float(lat.graph[e]), float(lat.acoustic[e]),
             int(lat.dur[e])) for e in keep]
    return arcs, fin, len(keep) < lat.narcs


@pytest.mark.parametrize("g", GROUPS)
def test_log_sweeps_with_beam(klu, ora, engine, monkeypatch, g):
    """The BEAM = true sweeps (run by the index tools under --beam): per state against the
    oracle on the lattice PruneLattice leaves (arcs and finals off, state ids kept)."""
    monkeypatch.setenv("KLU_SWEEP_LANES", str(g))
    lats = [lat for lat in adversarial(klu, g, seed=7) if lat.key != "range"]
    batch = klu.LatticeBatch.from_lattices(lats)
    engine.load(batch)
    for flags, beam in ((dict(), 4.0), (dict(acoustic_scale=0.1), 1.5),
                        (dict(graph_scale=0.7, insertion_penalty=0.5), 3.0)):
        engine.run(klu.SEGMENT, beam=beam, **flags)
        al, be, tot = engine.fetch_fwd_bwd()
        pruned_some = False
        for l, lat in enumerate(lats):
            arcs, fin, cut = _host_prune(lat, beam, flags)
            pruned_some |= cut
            p = klu.make_lattice(lat.key, lat.nstates, arcs, fin)
            a, b = int(batch.state_off[l]), int(batch.state_off[l + 1])
            check_states((al[a:b], be[a:b], tot[l]), ora.fwd_bwd(p, **flags),
                         "G=%d beam %g %r lattice %s" % (g, beam, flags, lat.key))
        assert pruned_some


def test_two_term_states_bit_identical_across_widths(klu, engine, monkeypatch):
    """Where every state has at most two terms the sweeps use Kaldi's LogAdd only: alpha,
    beta and total do not depend on the lane width, bit for bit."""
    rng = np.random.RandomState(3)
    lats = [diamond_lattice(klu, rng, 30 + 7 * i) for i in range(5)]
    lats.append(build(klu, "chain", 300, [(i, i + 1, *rng.uniform(0, 3, 2)) for i in range(299)], {299: (0.1, 0.2)}))
    batch = klu.LatticeBatch.from_lattices(lats)
    ref = None
    for g in GROUPS:
        monkeypatch.setenv("KLU_SWEEP_LANES", str(g))
        res = run_fwd_bwd(klu, engine, batch, acoustic_scale=0.1)
        if ref is None:
            ref = res
        for x, y in zip(ref, res):
            assert np.array_equal(x.view(np.int64), y.view(np.int64)), "G=%d differs from G=%d" % (g, GROUPS[0])


def test_automatic_width_at_scale(klu, ora, engine, monkeypatch):
    """test_alpha_beta_per_state's shapes once more in a batch large enough that
    run_log_sweeps picks G = 16 itself (the production width), a sample per state."""
    import torch
    monkeypatch.delenv("KLU_SWEEP_LANES", raising=False)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = sms * 8 + 64  # 2 L G / 32 >= 8 SMs first at G = 16
    base = (klu.synth_batch("tiny", 24, seed=5).lattices() + klu.synth_batch("small", 12, seed=6).lattices() +
            klu.synth_batch("c2", 3, seed=9).lattices())
    lats = [base[i % len(base)] for i in range(n)]
    batch = klu.LatticeBatch.from_lattices(lats)
    engine.load(batch)
    st = engine.stats()
    G = 4  # run_log_sweeps' choice, restated
    while G < 32 and G * 6 < st["arcs"] / st["levels"]:
        G <<= 1
    while G < 32 and 2 * n * G // 32 < sms * 8:
        G <<= 1
    assert G == 16, "the batch should take the production width, got %d" % G
    sample = sorted(set(range(len(base))) | set(np.random.RandomState(1).choice(n, 40, replace=False).tolist()))
    for flags in FLAGS:
        engine.run(klu.FWD_BWD, **flags)
        check_batch(ora, batch, engine.fetch_fwd_bwd(), flags, "auto G=16 %r" % flags, only=sample)


# ---- 3. tropical sweeps at every pick_group width ------------------------------------------------
def fanout_lattice(klu, rng, key, width, nlev, deg, ties):
    """start -> nlev levels of `width` states -> final.  Every state of a level but the last
    sends `deg` arcs to the next level (parallel arcs), the first of them to the state with
    its own index there.  With `ties`, every other arc has a twin with the same weights and
    another label: paths of exactly equal cost."""
    lvl = [list(range(1 + k * width, 1 + (k + 1) * width)) for k in range(nlev)]
    fin = 1 + nlev * width
    arcs = [(0, s, *rng.uniform(0, 2, 2), 0) for s in lvl[0]]
    for k in range(nlev - 1):
        for i, s in enumerate(lvl[k]):
            for e in range(deg):
                d = lvl[k + 1][i] if e == 0 else int(rng.choice(lvl[k + 1]))
                g, a = float(np.float32(rng.uniform(0, 4))), float(np.float32(rng.uniform(0, 4)))
                lab = int(rng.randint(1, 6)) if rng.rand() < 0.4 else 0
                arcs.append((s, d, g, a, lab))
                if ties and e % 2 == 1:
                    arcs.append((s, d, g, a, lab % 5 + 1))
    arcs += [(s, fin, float(rng.uniform(0, 2)), 0.5, 0) for s in lvl[-1]]
    return build(klu, key, fin + 1, arcs, {fin: (0.25, 0.0)})


BANDS = [(2.5, 2), (5.0, 4), (20.0, 8), (100.0, 16), (200.0, 32)]


def fanout_batch(klu, target):
    """Six fan-out lattices (three with cost ties) whose arcs per state, over the batch, come
    closest to `target`."""
    best = None
    for deg in range(1, int(target) + 3):
        rng = np.random.RandomState(int(target * 10))
        lats = [fanout_lattice(klu, rng, "fan%d" % i, width=4 + i % 3, nlev=5, deg=deg, ties=i % 2 == 1)
                for i in range(6)]
        batch = klu.LatticeBatch.from_lattices(lats)
        mean = batch.num_arcs / batch.num_states
        if best is None or abs(mean - target) < abs(best[2] - target):
            best = (lats, batch, mean)
    return best


@pytest.mark.parametrize("target,group", BANDS, ids=["deg%g" % t for t, _ in BANDS])
def test_tropical_sweeps_each_width(klu, ora, engine, target, group):
    """Batches whose arcs per state fall in each pick_group band (means 2.3, 5.0, 20.3, 99.9
    and 199.5): lattice-prune-dyn-beam (arcs, weights, beams bit-exact) and
    lattice-best-path2 (labels bit-exact) against the oracle."""
    lats, batch, mean = fanout_batch(klu, target)
    assert pick_group(mean) == group, "mean degree %.2f lands in the band of G=%d" % (mean, pick_group(mean))
    engine.load(batch)
    flags = dict(max_arcs=int(batch.num_arcs / len(lats) / 3), max_states=1000, beam_ratio=0.8)
    got = engine.prune_dyn_beam(**flags)
    for l, lat in enumerate(lats):
        w = ora.prune_dyn_beam(lat, **flags)
        assert got[l]["nstates"] == w["nstates"] and got[l]["arcs"] == w["arcs"] and got[l]["finals"] == w["finals"], \
            "prune-dyn-beam, lattice %d (mean degree %.1f)" % (l, mean)
        assert got[l]["beam0"] == w["beam0"] and got[l]["beam"] == w["beam"]
    for flags in (dict(), dict(acoustic_scale=0.1)):
        bp = engine.best_path2(**flags)
        for l, lat in enumerate(lats):
            labels, cost = ora.best_path2(lat, **flags)
            assert bp[l][0] == labels, "best-path2 labels, lattice %d (mean degree %.1f)" % (l, mean)
            assert abs(bp[l][1] - cost) <= 1e-4 * max(1.0, abs(cost))


# ---- 4. k_banded_alpha pieces ---------------------------------------------------------------
def band_lattice(klu, rng, key, width=None, in_counts=None):
    """start -> a level of `width` states -> (optionally) states with the given in-arc counts
    from that level -> final.  Labels on the first two hops only: at most 3 distinct lengths."""
    width = width or 12
    first = 1
    lvl1 = list(range(first, first + width))
    arcs = [(0, s, *rng.uniform(0, 2, 2), int(rng.randint(0, 4))) for s in lvl1]
    nxt = first + width
    lvl2 = []
    for k, cnt in enumerate(in_counts or []):
        s = nxt + k
        lvl2.append(s)
        arcs.append((lvl1[0], s, *rng.uniform(0, 3, 2), int(rng.randint(1, 5))))
        arcs += [(int(rng.choice(lvl1)), s, *rng.uniform(0, 3, 2), int(rng.randint(0, 5))) for _ in range(cnt - 1)]
    f = nxt + len(lvl2)
    ends = lvl2 if lvl2 else lvl1
    arcs += [(s, f, *rng.uniform(0, 2, 2), 0) for s in ends]
    if lvl2:
        arcs += [(s, f, *rng.uniform(0, 2, 2), 0) for s in lvl1[::5]]
    return build(klu, key, f + 1, arcs, {f: (0.0, 0.5), lvl1[1]: (1.0, 0.0)})


def band_lattices(klu):
    rng = np.random.RandomState(17)
    lats = [band_lattice(klu, rng, "w%d" % w, width=w) for w in (BAND_STATES - 1, BAND_STATES, BAND_STATES + 1)]
    for total in (BAND_ARCS - 1, BAND_ARCS, BAND_ARCS + 1):
        k = 8
        counts = [total // k] * (k - 1)
        counts.append(total - sum(counts))
        lats.append(band_lattice(klu, rng, "a%d" % total, width=20, in_counts=counts))
    # one state with more in-arcs than a piece stages, between ordinary ones
    lats.append(band_lattice(klu, rng, "big", width=24, in_counts=[5, BAND_ARCS + 40, 7]))
    return lats


@pytest.mark.parametrize("flags", [dict(), dict(acoustic_scale=0.1), dict(acoustic_scale=0.1, beam=3.0)],
                         ids=["plain", "ac0.1", "beam"])
def test_banded_alpha_pieces(klu, ora, engine, monkeypatch, flags):
    """Levels of 127 / 128 / 129 states, levels with 767 / 768 / 769 in-arcs and one state over
    768 (the not-staged path): lattice-word-index-position and lattice-to-word-position-post
    against the oracle at 1e-4, and the position rows of the generic path
    (KLU_GENERIC_POSITION=1) against the default one at 1e-9."""
    lats = band_lattices(klu)
    batch = klu.LatticeBatch.from_lattices(lats)
    engine.load(batch)
    monkeypatch.delenv("KLU_GENERIC_POSITION", raising=False)
    got = engine.position(**flags)
    for l, lat in enumerate(lats):
        assert_rows_match(got[l], ora.position(lat, **flags), 2, what="position %s %r" % (lat.key, flags))
    monkeypatch.setenv("KLU_GENERIC_POSITION", "1")
    gen = engine.position(**flags)
    monkeypatch.delenv("KLU_GENERIC_POSITION")
    for l, lat in enumerate(lats):
        gm, dm = {r[:4]: r[-1] for r in gen[l]}, {r[:4]: r[-1] for r in got[l]}
        assert gm.keys() == dm.keys(), "generic position keys, %s" % lat.key
        for k, v in dm.items():
            assert abs(gm[k] - v) <= 1e-9 * max(1.0, abs(v)), "generic position %s %s: %r vs %r" % (lat.key, k, gm[k], v)
    if "beam" in flags:
        return  # position-post takes no beam
    pp = engine.position_post(**flags)
    for l, lat in enumerate(lats):
        want = ora.position_post(lat, **flags)
        assert len(pp[l]) == len(want), "position-post positions, %s" % lat.key
        for p, (g, w) in enumerate(zip(pp[l], want)):
            assert dict(g).keys() == dict(w).keys(), "position-post words, %s position %d" % (lat.key, p)
            for wd, v in w:
                assert abs(dict(g)[wd] - v) <= 1e-4, "position-post %s position %d word %d" % (lat.key, p, wd)


# ---- 5. fast_exp / fast_log / log_add on the device ---------------------------------------------
PROBE = r"""
#include <stdio.h>
#include <vector>
#include "klu_common.cuh"

__global__ void k_probe(const double* x, const double* y, int n, double* ex, double* lg, double* la) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ex[i] = klu::fast_exp(x[i]);
  lg[i] = x[i] > 0.0 ? klu::fast_log(x[i]) : 0.0;
  la[i] = klu::log_add(x[i], y[i]);
}

int main(int argc, char** argv) {
  FILE* f = fopen(argv[1], "rb");
  long n = 0;
  fseek(f, 0, SEEK_END);
  n = ftell(f) / 16;
  fseek(f, 0, SEEK_SET);
  std::vector<double> h(2 * n), out(3 * n);
  if (fread(h.data(), 16, n, f) != (size_t)n) return 2;
  fclose(f);
  double *d_in, *d_out;
  if (cudaMalloc(&d_in, 16 * n) != cudaSuccess || cudaMalloc(&d_out, 24 * n) != cudaSuccess) return 3;
  cudaMemcpy(d_in, h.data(), 16 * n, cudaMemcpyHostToDevice);
  k_probe<<<(n + 255) / 256, 256>>>(d_in, d_in + n, (int)n, d_out, d_out + n, d_out + 2 * n);
  if (cudaDeviceSynchronize() != cudaSuccess) return 4;
  cudaMemcpy(out.data(), d_out, 24 * n, cudaMemcpyDeviceToHost);
  f = fopen(argv[2], "wb");
  fwrite(out.data(), 8, 3 * n, f);
  fclose(f);
  cudaFree(d_in);
  cudaFree(d_out);
  return 0;
}
"""


def _nvflags():
    """NVFLAGS of the package Makefile (the flags the library is compiled with)."""
    text = open(os.path.join(PKG, "Makefile")).read()
    return re.search(r"^NVFLAGS \?= (.*)$", text, re.M).group(1).split()


def _bits(h, lo):
    return np.array([(int(h) << 32) | int(lo)], np.uint64).view(np.float64)[0]


def test_fast_exp_log_log_add_bounds(tmp_path):
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    src = tmp_path / "probe.cu"
    src.write_text(PROBE)
    exe = tmp_path / "probe"
    subprocess.run([nvcc] + _nvflags() + ["-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(PKG, "csrc"),
                    str(src), "-o", str(exe)], check=True, capture_output=True)
    rng = np.random.RandomState(11)
    ulp700 = np.spacing(700.0)
    xe = np.concatenate([np.linspace(-700.0, 700.0, 400001), rng.uniform(-700, 700, 200000), rng.normal(0, 5, 50000),
                         [700.0, -700.0, 700.0 - ulp700, -700.0 + ulp700, 700.0 + ulp700, -700.0 - ulp700,
                          np.inf, -np.inf, np.nan, 0.0, -0.0]])
    split = _bits(0x3ff6a09f, 0)
    xl = np.concatenate([np.ldexp(1.0, np.arange(-1022, 1024)),
                         np.ldexp(np.array([np.nextafter(split, 0), split, np.nextafter(split, 2)])[:, None],
                                  np.arange(-1000, 1001, 37)[None, :]).ravel(),
                         [1e-280, 1e280, 1.0, np.nextafter(1.0, 2), np.nextafter(1.0, 0)],
                         np.ldexp(rng.uniform(1, 2, 100000), rng.randint(-1021, 1023, 100000)),
                         rng.uniform(0.5, 2.0, 100000)])
    cut = -36.04365338911715
    xa = rng.normal(0, 50, 100000)
    ya = xa + np.concatenate([rng.uniform(-40, 40, 99000), np.full(1000, cut)])
    edge_x = np.array([0.0, 0.0, 0.0, 0.0, 1.0, -np.inf, -np.inf, 3.0, 5.0])
    edge_y = np.array([cut, np.nextafter(cut, -np.inf), np.nextafter(cut, 0), -50.0, 1.0, -np.inf, 3.0, -np.inf, 5.0 + cut])
    x = np.concatenate([xe, xl, xa, edge_x])
    y = np.concatenate([np.zeros(len(xe) + len(xl)), ya, edge_y])
    inp = tmp_path / "in.bin"
    np.concatenate([x, y]).astype(np.float64).tofile(str(inp))
    outp = tmp_path / "out.bin"
    subprocess.run([str(exe), str(inp), str(outp)], check=True)
    out = np.fromfile(str(outp), np.float64).reshape(3, len(x))
    ex, lg, la = out

    # exp: relative < 1e-14 inside the guard; 0 below, +inf above and for NaN
    e = ex[:len(xe)]
    inside = np.abs(xe) <= 700.0
    ref = np.exp(xe[inside].astype(np.longdouble))
    rel = np.abs((e[inside].astype(np.longdouble) - ref) / ref).astype(np.float64)
    k = int(np.argmax(rel))
    assert rel[k] < 1e-14, "fast_exp(%r): relative error %g" % (xe[inside][k], rel[k])
    assert (e[inside] > 0).all() and np.isfinite(e[inside]).all()
    out_lo = (xe < -700.0) & ~np.isnan(xe)
    out_hi = (xe > 700.0) | np.isnan(xe)
    assert (e[out_lo] == 0.0).all() and np.isposinf(e[out_hi]).all()

    # log: absolute < 1e-15 max(1, |log s|) on positive normals
    lgs = lg[len(xe):len(xe) + len(xl)]
    ref = np.log(xl.astype(np.longdouble))
    err = (np.abs(lgs.astype(np.longdouble) - ref) / np.maximum(1.0, np.abs(ref))).astype(np.float64)
    k = int(np.argmax(err))
    assert err[k] < 1e-15, "fast_log(%r): error %g relative to max(1, |log s|)" % (xl[k], err[k])

    # log_add: Kaldi's LogAdd restated on the host, within 2 ulp; exactly max below the cut.
    # CUDA's exp / log1p are not glibc's, and max + log1p(exp(d)) cancels when max < 0 (max
    # -0.83, log1p term +0.60, sum -0.23: one ulp of the operand is four of the sum), so the
    # ulp is taken at the larger of |max| and |result|.
    a0 = len(xe) + len(xl)
    xs, ys, got = x[a0:], y[a0:], la[a0:]
    with np.errstate(invalid="ignore", over="ignore"):
        hi, lo = np.maximum(xs, ys), np.minimum(xs, ys)
        diff = lo - hi
        use = diff >= cut
        want = np.where(use, hi + np.log1p(np.exp(np.where(use, diff, 0.0))), hi)
    both_inf = np.isneginf(xs) & np.isneginf(ys)
    assert np.isneginf(got[both_inf]).all()
    m = ~both_inf
    assert np.isfinite(got[m]).all() and np.isfinite(want[m]).all()
    du = np.abs(got[m] - want[m]) / np.spacing(np.maximum(np.abs(hi[m]), np.abs(want[m])))
    k = int(np.argmax(du))
    assert du[k] <= 2, "log_add(%r, %r) = %r, Kaldi %r: %g ulp" % (xs[m][k], ys[m][k], got[m][k], want[m][k], du[k])
    below = m & (diff < cut)
    assert np.array_equal(got[below], np.maximum(xs, ys)[below])
    assert got[len(xa) + 1] == 0.0 and got[len(xa)] > 0.0  # at the cut: log1p; one ulp below: max
