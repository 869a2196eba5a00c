"""Parity at the BASELINE shapes, wider than test_gpu_scale.py: the banded (state, length)
tools on 32 full c2 lattices, the utterance tool on deep c4 lattices, per-state alpha/beta,
prune -> best-path2 through the two binaries on 2000 c2 lattices, batches of more than 65535
lattices, klu_topsort feeding lattice-prune-dyn-beam, several GPUs through KLU_DEVICES.

The oracle runs on all host threads (ctypes releases the GIL); results are compared as numpy
columns (a c2 lattice has ~1.5 M position entries)."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from util import TOL, assert_cols_match, assert_rows_match

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "kaldi-lattice-utils_b200", "bin")


def _pool():
    return ThreadPoolExecutor(max_workers=max(1, min(os.cpu_count() or 1, 32)))


# ---- alpha / beta per state -------------------------------------------------------------
@pytest.mark.parametrize("shape,n,seed", [("tiny", 24, 5), ("small", 12, 6), ("c2", 3, 9)])
@pytest.mark.parametrize("flags", [dict(), dict(acoustic_scale=0.1), dict(graph_scale=0.7, insertion_penalty=0.5)])
def test_alpha_beta_per_state(klu, ora, engine, shape, n, seed, flags):
    """ComputeLatticeAlphasAndBetas [ext]: every state's alpha and beta (input numbering) and
    the returned 0.5 * (tot_fwd + beta[0]), not just the total."""
    batch = klu.synth_batch(shape, n, seed=seed)
    engine.load(batch)
    engine.run(klu.FWD_BWD, **flags)
    al, be, tot = engine.fetch_fwd_bwd()
    for l, lat in enumerate(batch.lattices()):
        a, b = int(batch.state_off[l]), int(batch.state_off[l + 1])
        wa, wb, wt = ora.fwd_bwd(lat, **flags)
        assert np.array_equal(np.isinf(al[a:b]), np.isinf(wa)) and np.array_equal(np.isinf(be[a:b]), np.isinf(wb))
        fin = np.isfinite(wa) & np.isfinite(wb)
        assert np.abs(al[a:b][fin] - wa[fin]).max() <= 1e-9 * max(1.0, np.abs(wa[fin]).max())
        assert np.abs(be[a:b][fin] - wb[fin]).max() <= 1e-9 * max(1.0, np.abs(wb[fin]).max())
        assert abs(tot[l] - wt) <= 1e-9 * max(1.0, abs(wt))


# ---- the banded tools on 32 full c2 lattices -----------------------------------------------
def test_c2_position_family_32_lattices(klu, ora, engine):
    """lattice-word-index-position, lattice-best-path2 and lattice-to-word-position-post on 32
    c2 lattices (~1.5 M (word, position) entries each), every row against the oracle."""
    n = 32
    flags = dict(acoustic_scale=0.1)
    batch = klu.synth_batch("c2", n, seed=21)
    lats = batch.lattices()
    with _pool() as ex:
        want_pos = [ex.submit(ora.run, ora.POSITION, lat, **flags) for lat in lats]
        want_bp = [ex.submit(ora.best_path2, lat, **flags) for lat in lats]
        want_pp = [ex.submit(ora.run, ora.POSITION_POST, lat, **flags) for lat in lats]
        engine.load(batch)
        engine.run(klu.POSITION, **flags)
        off, w, p, t0, t1, lp = engine.fetch_position()
        for l in range(n):
            r = want_pos[l].result()
            want_pos[l] = None
            a, b = int(off[l]), int(off[l + 1])
            assert_cols_match((w[a:b], p[a:b]), (t0[a:b], t1[a:b]), lp[a:b], (r.i[0], r.i[1]), (r.i[2], r.i[3]), r.d,
                              what="c2 position lat %d" % l)
        del off, w, p, t0, t1, lp
        engine.run(klu.BEST_PATH2, **flags)
        off, lab, cost, nf = engine.fetch_best_path2()
        for l in range(n):
            labels, c = want_bp[l].result()
            assert lab[int(off[l]):int(off[l + 1])].tolist() == labels, "best-path2 labels, lattice %d" % l
            assert abs(float(cost[l]) - c) <= 1e-4 * max(1.0, abs(c))
        engine.run(klu.POSITION_POST, **flags)
        off, npos, pos, w, lp = engine.fetch_position_post()
        for l in range(n):
            r = want_pp[l].result()
            want_pp[l] = None
            a, b = int(off[l]), int(off[l + 1])
            assert int(npos[l]) == r.s0
            # rows are grouped by position (ascending), inside a position by (float logp desc, word)
            assert (np.diff(pos[a:b]) >= 0).all()
            assert_cols_match((pos[a:b], w[a:b]), (), lp[a:b].astype(np.float64), (r.i[0], r.i[1]), (),
                              r.f[0].astype(np.float64), what="c2 position-post lat %d" % l, ordered=False)


# ---- utterance at the c4 shape ----------------------------------------------------------------
def test_c4_utterance_deep_lattices(klu, ora, engine):
    """lattice-word-index-utterance on deep lattices (~20k states, ~500k arcs).  The reference
    composes the lattice with a query automaton per word, so the oracle needs minutes per
    lattice for all ~40k words: 64 words per lattice (the most frequent, the rarest and random
    ones) are checked against it through --include-words, and the full run must agree with the
    filtered one on those words."""
    batch = klu.synth_batch("c4", 2, seed=7)
    lats = batch.lattices()
    engine.load(batch)
    full = engine.utterance(acoustic_scale=0.1)
    rng = np.random.RandomState(4)
    for l, lat in enumerate(lats):
        words, counts = np.unique(lat.label[lat.label != 0], return_counts=True)
        by_freq = words[np.argsort(-counts, kind="stable")]
        sample = sorted(set(by_freq[:16].tolist()) | set(by_freq[-16:].tolist()) |
                        set(rng.choice(words, 32, replace=False).tolist()))
        one = klu.LatticeBatch.from_lattices([lat])
        engine.load(one)
        got = engine.utterance(acoustic_scale=0.1, include_words=sample)[0]
        want = ora.utterance(lat, acoustic_scale=0.1, include_words=sample)
        assert_rows_match(got, want, 1, what="c4 utterance lat %d" % l)
        fm = dict(full[l])
        assert len(full[l]) == len(words)
        for wd, v in got:
            assert fm[wd] == v  # same arithmetic with and without the filter
        vals = [v for _, v in full[l]]
        assert all(x >= y for x, y in zip(vals[:-1], vals[1:])) and max(vals) <= 1e-9


# ---- more than 65535 lattices in one batch ---------------------------------------------------
def test_batch_of_70000_lattices(klu, ora, engine):
    """The library has no per-batch lattice limit (lattices ride blockIdx.x)."""
    base = klu.synth_batch("tiny", 7, seed=3).lattices()
    n = 70000
    batch = klu.LatticeBatch.from_lattices([base[i % 7] for i in range(n)])
    engine.load(batch)
    want = [ora.segment(lat) for lat in base]
    wantp = [ora.position(lat) for lat in base]
    engine.run(klu.SEGMENT)
    off, w, t0, t1, lp = engine.fetch_segment()
    assert len(off) == n + 1
    for l in (0, 1, 6, 65534, 65535, 65536, 65537, n - 1):
        a, b = int(off[l]), int(off[l + 1])
        got = list(zip(w[a:b].tolist(), t0[a:b].tolist(), t1[a:b].tolist(), lp[a:b].tolist()))
        assert_rows_match(got, want[l % 7], 3, what="lattice %d of 70000" % l)
    # every copy of a lattice gives bit-identical rows
    for l in range(7, n, 997):
        a, b, a0, b0 = int(off[l]), int(off[l + 1]), int(off[l % 7]), int(off[l % 7 + 1])
        assert b - a == b0 - a0 and np.array_equal(lp[a:b], lp[a0:b0]) and np.array_equal(w[a:b], w[a0:b0])
    engine.run(klu.POSITION)
    off, w, p, t0, t1, lp = engine.fetch_position()
    for l in (0, 65535, 65536, n - 1):
        a, b = int(off[l]), int(off[l + 1])
        got = list(zip(w[a:b].tolist(), p[a:b].tolist(), t0[a:b].tolist(), t1[a:b].tolist(), lp[a:b].tolist()))
        assert_rows_match(got, wantp[l % 7], 2, what="position, lattice %d of 70000" % l)
    engine.run(klu.FRAME_POST)
    foff = engine.fetch_frame_post()[0]
    assert len(foff) == n + 1 and (np.diff(foff) > 0).all()


# ---- klu_topsort -> lattice-prune-dyn-beam: state ids as the reference would write them ----------
def test_topsort_then_prune_matches_oracle(klu, ora, engine):
    """Lattices with shuffled state ids: klu_topsort numbers the states, lattice-prune-dyn-beam
    writes them; both must equal the oracle's fst::TopSort restatement followed by its
    PruneDynBeam (arcs, new state ids, weights bit-exact)."""
    from test_topsort import _apply_order, _call

    def connected_dag(n):
        # every state reachable from the start and on a path to the final state (the reference's
        # pruning loop does not terminate on anything else: infinite lattice beam)
        arcs = []
        for s in range(1, n):
            for p in set([int(rng.randint(max(0, s - 3), s))] + [int(rng.randint(max(0, s - 6), s)) for _ in range(2)]):
                arcs.append((p, s, int(rng.randint(0, 6)), float(rng.uniform(0, 3)), float(rng.uniform(0, 3)), s - p))
        for s in range(n - 1):
            if not any(a[0] == s for a in arcs):
                arcs.append((s, s + 1, 1, 1.0, 1.0, 1))
        perm = np.arange(n)
        perm[1:] = rng.permutation(np.arange(1, n))
        arcs = [(int(perm[u]), int(perm[v]), w, g, a, t) for (u, v, w, g, a, t) in arcs]
        arcs.sort(key=lambda x: x[0])
        return klu.make_lattice("dag", n, arcs, {int(perm[n - 1]): (0.5, 0.25)})

    rng = np.random.RandomState(77)
    sorted_lats, want = [], []
    for k in range(10):
        lat = connected_dag(20 + 5 * k)
        rc, got, order = _call(klu, lat)
        assert rc == 0 and order.tolist() == ora.top_order(lat)
        s = _apply_order(klu, lat, order.tolist())
        for f in ("src", "dst", "label", "dur"):
            assert np.array_equal(got[f], getattr(s, f))
        sorted_lats.append(s)
    flags = dict(max_arcs=25, max_states=18, beam_ratio=0.8)
    engine.load(klu.LatticeBatch.from_lattices(sorted_lats))
    got = engine.prune_dyn_beam(**flags)
    for l, s in enumerate(sorted_lats):
        w = ora.prune_dyn_beam(s, **flags)
        assert got[l]["nstates"] == w["nstates"] and got[l]["arcs"] == w["arcs"] and got[l]["finals"] == w["finals"]
        assert got[l]["beam0"] == w["beam0"] and got[l]["beam"] == w["beam"]


# ---- configs[2] through the binaries -------------------------------------------------------------
def _synth_ark(klu, path, shape, n, seed):
    cfg = klu.lattice.SHAPES[shape]
    subprocess.run([os.path.join(BIN, "klu-synth-lattices")] + [str(cfg[k]) for k in (
        "frames", "states_per_frame", "arcs_per_state", "max_skip", "vocab", "pool_size", "window", "eps_prob",
        "weight_max", "kind")] + [str(seed), str(n), "ark:" + path], check=True)


def test_c3_prune_then_best_path2_through_the_binaries(klu, ora, tmp_path):
    """BASELINE.json configs[2]: lattice-prune-dyn-beam --max-arcs=20000 --max-states=1500
    --beam-ratio=0.9 piped into lattice-best-path2, 2000 c2 lattices, both as processes.  Every
    utterance must come out, in input order; 48 of them are recomputed by the oracle (prune, then
    best-path2 on the pruned lattice) and must give the same label sequence."""
    n, seed = 2000, 33
    ark = str(tmp_path / "c2.ark")
    _synth_ark(klu, ark, "c2", n, seed)
    out = str(tmp_path / "best.txt")
    prune = [os.path.join(BIN, "lattice-prune-dyn-beam"), "--max-arcs=20000", "--max-states=1500",
             "--beam-ratio=0.9", "ark:" + ark, "ark:-"]
    best = [os.path.join(BIN, "lattice-best-path2"), "ark:-", "ark,t:" + out]
    # (the tools log one line per lattice: stderr goes to files, an unread pipe would fill up)
    with open(str(tmp_path / "prune.err"), "wb") as e1, open(str(tmp_path / "best.err"), "wb") as e2:
        p1 = subprocess.Popen(prune, stdout=subprocess.PIPE, stderr=e1)
        p2 = subprocess.Popen(best, stdin=p1.stdout, stderr=e2)
        p1.stdout.close()
        p2.wait()
        p1.wait()
    assert p1.returncode == 0, open(str(tmp_path / "prune.err")).read()[-2000:]
    assert p2.returncode == 0, open(str(tmp_path / "best.err")).read()[-2000:]
    lines = open(out).read().strip("\n").split("\n")
    assert [x.split()[0] for x in lines] == ["utt%07d" % i for i in range(n)]
    os.remove(ark)
    pick = sorted(np.random.RandomState(5).choice(n, 48, replace=False).tolist())
    flags = dict(max_arcs=20000, max_states=1500, beam_ratio=0.9)

    def oracle_pipe(l):
        lat = klu.synth_batch("c2", 1, seed=seed, first_id=l)[0]
        p = ora.prune_dyn_beam(lat, **flags)
        arcs = [(s, d, lab, g, a, int(lat.dur[i])) for i, s, d, lab, g, a in p["arcs"]]
        finals = {s: (g, a) for s, g, a in p["finals"]}
        return ora.best_path2(klu.make_lattice(lat.key, p["nstates"], arcs, finals))[0]

    with _pool() as ex:
        want = list(ex.map(oracle_pipe, pick))
    for l, labels in zip(pick, want):
        assert [int(x) for x in lines[l].split()[1:]] == labels, "utterance %d" % l


# ---- several GPUs through the tools' own partitioner ------------------------------------------------
@pytest.mark.parametrize("tool,args", [("lattice-word-index-segment", []), ("lattice-to-word-frame-post", []),
                                       ("lattice-prune-dyn-beam", ["--max-arcs=400"])])
def test_klu_devices_on_several_gpus(klu, tmp_path, tool, args):
    """KLU_DEVICES=0,1,...: one worker thread + context per GPU takes batches in turn; the
    output must be byte-identical to the one-GPU run (P9: entries in input order)."""
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("one GPU")
    ark = str(tmp_path / "small.ark")
    _synth_ark(klu, ark, "small", 600, 11)
    env1 = dict(os.environ, KLU_DEVICES="0", KLU_BATCH_ARCS="20000")
    envn = dict(os.environ, KLU_DEVICES=",".join(str(i) for i in range(ngpu)), KLU_BATCH_ARCS="20000")
    one = subprocess.run([os.path.join(BIN, tool)] + args + ["ark:" + ark, "ark:-"], capture_output=True, env=env1)
    many = subprocess.run([os.path.join(BIN, tool)] + args + ["ark:" + ark, "ark:-"], capture_output=True, env=envn)
    assert one.returncode == 0 and many.returncode == 0, many.stderr.decode()[-2000:]
    assert len(one.stdout) > 100000 and many.stdout == one.stdout


# ---- the multi-CTA sort passes (klu_sort.cuh) on the whole parity suite --------------------------
def test_parity_suite_with_multi_cta_sorts(tmp_path):
    """seg_sort_launch picks the multi-CTA passes only for large segments, which the small parity
    shapes never reach: run the parity tests of every tool that sorts once more with
    KLU_SORT_MULTI=1 (the switch is read once per process, hence the child process)."""
    env = dict(os.environ, KLU_SORT_MULTI="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    log = tmp_path / "multi_sort_suite.log"
    with open(str(log), "w") as f:
        rc = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_parity.py"),
                             os.path.join(root, "tests", "test_gpu_char.py"), "-m", "gpu", "-x", "-q",
                             "--timeout", "300", "--timeout-method", "thread", "-p", "no:cacheprovider"],
                            env=env, cwd=root, stdout=f, stderr=subprocess.STDOUT, timeout=900).returncode
    assert rc == 0, "parity suite failed with KLU_SORT_MULTI=1:\n" + log.read_text()[-3000:]
