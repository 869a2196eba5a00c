"""The static frame index of the frame-synchronous word posteriorgram (klu_frame.cu) on
batches built to reach each of its layouts: lattices crowded with arcs that have no
arc x frame instance, windows too long for shared memory, ids wider than 16 bits, and
groups whose posterior sum underflows.  Each batch restates the condition it relies on
and is checked against the oracle and against the generic pipeline."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FRAMES_PER_RUN = 16  # kFramesPerItem
WIN_CAP = 8192       # windows longer than this (64 KB of f64 posteriors) take the path without shared memory


def arc_frames(lat):
    """(start frame, end frame, spans a frame as a word arc) per arc, and the frame count.
    State ids of these lattices are topologically sorted (src < dst)."""
    t = np.zeros(lat.nstates, np.int64)
    for i in np.argsort(lat.src, kind="stable"):
        t[lat.dst[i]] = t[lat.src[i]] + lat.dur[i]
    fin = np.isfinite(lat.fin_graph)
    T = int((t[fin] + lat.fin_dur[fin]).max())
    fa, fb = t[lat.src], np.minimum(t[lat.dst], T)
    return fa, fb, (lat.label != 0) & (fb > fa), T


def runs(lat):
    """Per run of frames: the fewest and the most arcs its window can hold (ties in start
    frame are ordered by the packed arc order), and how many arcs without an instance
    start inside its window's frame range."""
    fa, fb, word, T = arc_frames(lat)
    out = []
    for k0 in range(0, T, FRAMES_PER_RUN):
        k1 = min(T, k0 + FRAMES_PER_RUN)
        alive = word & (fa < k1) & (fb > k0)
        if not alive.any():
            continue
        lo, hi = fa[alive].min(), fa[alive].max()
        inner = word & (fa > lo) & (fa < hi)
        out.append(dict(least=int((alive | inner).sum()), most=int((word & (fa >= lo) & (fa <= hi)).sum()),
                        others=int((~word & (fa >= lo) & (fa <= hi)).sum()), words=int(alive.sum())))
    return out


def sausage(klu, key, T, per_frame, rng, long_arc=False, eps=0, zero_dur=0, unlikely=None):
    """T frames, one state per frame boundary (states 2k) with a side state (2k + 1) in
    between.  Per frame: `per_frame` word arcs of one frame, `eps` epsilon arcs of one frame,
    `zero_dur` word arcs into the side state that span no frame (the side state goes on with
    an epsilon arc).  `long_arc`: one word arc over the whole utterance.  `unlikely`: per
    frame one more arc, of word 5000 + frame, that many nats worse than the frame's best."""
    arcs = []
    for k in range(T):
        u, v, side = 2 * k, 2 * k + 2, 2 * k + 1
        costs = rng.uniform(0, 3, size=(per_frame, 2)).astype(np.float32)
        for i in range(per_frame):
            arcs.append((u, v, int(rng.randint(1, 150)), float(costs[i, 0]), float(costs[i, 1]), 1))
        for _ in range(eps):
            arcs.append((u, v, 0, float(rng.uniform(0, 3)), float(rng.uniform(0, 3)), 1))
        for _ in range(zero_dur):
            arcs.append((u, side, int(rng.randint(1, 150)), float(rng.uniform(0, 3)), 0.0, 0))
        if zero_dur:
            arcs.append((side, v, 0, 0.5, float(rng.uniform(0, 3)), 1))
        if unlikely is not None:
            arcs.append((u, v, 5000 + k, float((costs.sum(1)).min()) + unlikely, 0.0, 1))
    if long_arc:
        arcs.append((0, 2 * T, 7, 1.0, 2.0 * T, T))
    return klu.make_lattice(key, 2 * T + 1, arcs, {2 * T: (0.0, 0.0)})


def assert_frames_match(got, want, tol, what):
    assert len(got) == len(want), what
    for k, (g, w) in enumerate(zip(got, want)):
        gm, wm = dict(g), dict(w)
        assert len(gm) == len(g) and gm.keys() == wm.keys(), "%s frame %d: words differ" % (what, k)
        for word, b in wm.items():
            assert abs(gm[word] - b) <= tol * max(1.0, abs(b)), "%s frame %d word %d: %r vs %r" % (what, k, word, gm[word], b)
        for a, b in zip(g[:-1], g[1:]):  # the reference's order on our floats
            assert a[1] > b[1] or (a[1] == b[1] and a[0] < b[0]), "%s frame %d: order" % (what, k)


def check(klu, ora, engine, monkeypatch, lats):
    engine.load(klu.LatticeBatch.from_lattices(lats))
    fast = engine.frame_post()
    for l, lat in enumerate(lats):
        assert_frames_match(fast[l], ora.frame_post(lat), 1e-4, "%s vs oracle" % lat.key)
    monkeypatch.setenv("KLU_GENERIC_FRAME_POST", "1")
    generic = engine.frame_post()
    monkeypatch.delenv("KLU_GENERIC_FRAME_POST")
    for l, lat in enumerate(lats):
        assert_frames_match(fast[l], generic[l], 1e-6, "%s vs generic" % lat.key)


def test_batch_crowded_with_epsilon_and_zero_length_arcs(klu, ora, engine, monkeypatch):
    """Results only: that such arcs stay out of the windows is a matter of speed, not visible here."""
    rng = np.random.RandomState(11)
    lats = [sausage(klu, "eps%d" % i, 40 + 7 * i, 5, rng, eps=8, zero_dur=6) for i in range(3)]
    lats += klu.synth_batch("small", 3, seed=12).lattices()
    for lat in lats[:3]:
        for r in runs(lat):
            assert r["others"] > 2 * r["words"], "arcs without an instance should crowd every window"
    check(klu, ora, engine, monkeypatch, lats)


def test_window_longer_than_shared_memory(klu, ora, engine, monkeypatch):
    rng = np.random.RandomState(13)
    lats = [sausage(klu, "long", 64, 160, rng, long_arc=True)] + klu.synth_batch("small", 3, seed=14).lattices()
    w = [r for lat in lats for r in runs(lat)]
    assert max(r["least"] for r in w) > WIN_CAP, "some run should not fit shared memory"
    assert min(r["most"] for r in w) <= WIN_CAP, "some run should fit it"
    assert max(r["most"] for r in w) < 65536, "the batch should keep 16-bit ids"
    check(klu, ora, engine, monkeypatch, lats)


def test_window_of_65536_arcs_or_more(klu, ora, engine, monkeypatch):
    rng = np.random.RandomState(15)
    lats = [sausage(klu, "wide", 64, 1100, rng, long_arc=True)] + klu.synth_batch("small", 3, seed=16).lattices()
    w = [r for lat in lats for r in runs(lat)]
    assert max(r["least"] for r in w) >= 65536, "the batch should take 32-bit ids"
    assert min(r["most"] for r in w) <= WIN_CAP, "some run should fit shared memory"
    check(klu, ora, engine, monkeypatch, lats)


def test_underflowing_groups_in_and_out_of_shared_memory(klu, ora, engine, monkeypatch):
    rng = np.random.RandomState(17)
    lats = [sausage(klu, "under", 40, 5, rng, unlikely=800.0),
            sausage(klu, "under-long", 64, 160, rng, long_arc=True, unlikely=800.0)]
    for lat in lats:
        fa, _, _, T = arc_frames(lat)
        cost = (lat.graph + lat.acoustic).astype(np.float64)
        one = lat.dur == 1
        for k in range(T):
            seg = one & (fa == k)
            rare = seg & (lat.label == 5000 + k)
            # the group's posterior is at most its arc's share of the frame's parallel arcs
            share = -cost[rare][0] - np.logaddexp.reduce(-cost[seg])
            assert share < np.log(1e-280)
    assert max(r["least"] for r in runs(lats[1])) > WIN_CAP
    check(klu, ora, engine, monkeypatch, lats)
    got = engine.frame_post()
    assert all(dict(got[0][k])[5000 + k] < -700.0 for k in range(40))
