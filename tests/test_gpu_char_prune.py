"""The character tools' n-best frontier cut (klu_char.cu, "frontier cut"): lattices whose
unpruned pseudo-word frontier exceeds 2^24 trie nodes at one depth are indexed, and the
cut never changes a result."""
import heapq
import math
import os
import subprocess

import numpy as np
import pytest

from util import TOL, assert_rows_match

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WS = 1  # whitespace label


# ---- a character lattice with a closed-form index -----------------------------------------
# One state per frame boundary (state t = frame t's start, time t).  Frame t has two character
# arcs with labels private to the frame (2 + 2t, 3 + 2t) and one whitespace arc, all one frame
# long; state K is final with weight 0.  A pseudo-word is then a run [a, b) of character frames
# with whitespace (or the lattice's ends) around it; its label sequence fixes a, b and every
# frame's choice, and its position is one more than the words of the prefix [0, a).  So
#   P(key) = F_n(a) * prod_{t in [a, b)} p_t(c_t) * B(b) / Z
# with F_n(a) = mass of the prefixes [0, a) with n words that end in whitespace (a > 0),
# B(b) = mass of the suffixes after the run (whitespace at b, anything after; 1 at b = K) and
# Z = prod_t (p_t(c0) + p_t(c1) + p_t(ws)).

def chain_probs(K, seed):
    rng = np.random.RandomState(seed)
    p = np.zeros((K, 3))
    for t in range(K):
        major = rng.uniform(0.45, 0.65)
        minor = rng.uniform(0.04, 0.12)
        ws = rng.uniform(0.2, 0.4)
        p[t] = (major, minor, ws) if rng.rand() < 0.5 else (minor, major, ws)
    return p


def chain_lattice(klu, key, p):
    K = len(p)
    arcs = []
    for t in range(K):
        for j, lab in enumerate((2 + 2 * t, 3 + 2 * t, WS)):
            arcs.append((t, t + 1, lab, float(np.float32(-math.log(p[t, j]))), 0.0, 1))
    return klu.make_lattice(key, K + 1, arcs, {K: (0.0, 0.0)})


def lattice_costs(p):
    # the weights exactly as the lattice stores them (float32 costs)
    return np.array([[float(np.float32(-math.log(x))) for x in row] for row in p])


def closed_form_parts(p):
    """log F[n][a], log B[b], log Z, per-frame character log-probabilities."""
    K = len(p)
    lp = -lattice_costs(p)
    chars = np.logaddexp(lp[:, 0], lp[:, 1])
    tot = np.logaddexp(chars, lp[:, 2])
    # W[n][k] after t frames: k = 0 (start or whitespace last), 1 (character last)
    logF = np.full((K + 2, K + 1), -np.inf)
    W = np.full((K + 2, 2), -np.inf)
    W[0, 0] = 0.0
    logF[:, 0] = W[:, 0]
    for t in range(K):
        nw = np.full_like(W, -np.inf)
        nw[:, 0] = np.logaddexp(W[:, 0], W[:, 1]) + lp[t, 2]
        nw[1:, 1] = np.logaddexp(nw[1:, 1], W[:-1, 0] + chars[t])  # a new word
        nw[:, 1] = np.logaddexp(nw[:, 1], W[:, 1] + chars[t])       # the word goes on
        W = nw
        logF[:, t + 1] = W[:, 0]
    logB = np.zeros(K + 1)
    suffix = 0.0
    for b in range(K - 1, -1, -1):
        logB[b] = lp[b, 2] + suffix
        suffix += tot[b]
    logZ = float(np.sum(tot))
    return logF, logB, logZ, lp


def closed_form_rows(p, nbest, segment=False):
    """The nbest rows, best first: (string, pos, t0, t1, logp) or, segment, (string, t0, t1, logp).
    A best-first search over (n, a, b) and the frames' choices: a run's choices are independent,
    so its k-th best choice set comes from the sorted per-frame losses (include / swap the last)."""
    K = len(p)
    logF, logB, logZ, lp = closed_form_parts(p)
    if segment:
        logF = np.logaddexp.reduce(logF, axis=0)[None, :]
    best_c = np.argmax(lp[:, :2], axis=1)
    loss = np.abs(lp[:, 0] - lp[:, 1])
    heap = []
    for n in range(logF.shape[0]):
        for a in range(K):
            if not np.isfinite(logF[n, a]):
                continue
            run = 0.0
            for b in range(a + 1, K + 1):
                run += lp[b - 1, best_c[b - 1]]
                s = logF[n, a] + run + logB[b] - logZ
                order = tuple(sorted(range(a, b), key=lambda t: (loss[t], t)))
                heapq.heappush(heap, (-s, n, a, b, order, ()))
    rows = []
    want = nbest + 50  # a margin past the cut for the tie-break of the final order
    while heap and len(rows) < want:
        ns, n, a, b, order, swapped = heapq.heappop(heap)
        c = [int(best_c[t]) for t in range(a, b)]
        for i in swapped:
            c[order[i] - a] ^= 1
        string = "_".join(str(2 + 2 * t + c[t - a]) for t in range(a, b))
        if segment:
            rows.append((string, a, b, -ns))
        else:
            rows.append((string, n + 1, a, b, -ns))
        last = swapped[-1] if swapped else -1
        if last + 1 < len(order):
            nxt = order[last + 1]
            heapq.heappush(heap, (ns + loss[nxt], n, a, b, order, swapped + (last + 1,)))
            if swapped:
                heapq.heappush(heap, (ns + loss[nxt] - loss[order[last]], n, a, b, order, swapped[:-1] + (last + 1,)))
    rows.sort(key=lambda r: (-r[-1], r[0], r[1] if not segment else (r[1], r[2])))
    return rows[:nbest]


def unpruned_frontier(K):
    """Trie nodes per depth without the cut: a depth-d node is a (position, start, d + 1 choices)
    with a run of d + 1 frames that fits (position = words before + 1)."""
    per = []
    for d in range(K):
        n = 0
        for a in range(K - d):
            npos = a // 2 + 1  # words of a prefix [0, a) ending in whitespace: 0 .. ceil((a - 1) / 2)
            n += npos * 2 ** (d + 1)
        per.append(n)
    return per


def test_closed_form_matches_oracle_small(klu, ora):
    for seed in (1, 2):
        p = chain_probs(7, seed)
        lat = chain_lattice(klu, "small", p)
        for nbest in (1, 5, 100000):
            want = ora.char_position(lat, [WS], nbest=nbest)
            got = closed_form_rows(p, nbest)
            assert_rows_match(got, want, 2, what="closed form position nbest %d" % nbest)
            want = ora.char_segment(lat, [WS], nbest=nbest)
            got = closed_form_rows(p, nbest, segment=True)
            assert_rows_match(got, want, 3, what="closed form segment nbest %d" % nbest)
        # the unpruned frontier count of the small lattice against its row count (every node is a row)
        assert sum(unpruned_frontier(7)) == len(ora.char_position(lat, [WS], nbest=10 ** 9))


def write_text_ark(path, key, K, p):
    costs = lattice_costs(p)
    with open(path, "w") as f:
        f.write(key + "\n")
        for t in range(K):
            for j, lab in enumerate((2 + 2 * t, 3 + 2 * t, WS)):
                f.write("%d\t%d\t%d\t%d\t%r,0\n" % (t, t + 1, lab, lab, float(np.float32(costs[t, j]))))
        f.write("%d\t0,0\n\n" % K)


def parse_char_ark(text):
    key, rest = text.strip().split(" ", 1)
    rows = []
    for ent in rest.split(";"):
        f = ent.split()
        if f:
            rows.append((f[0], int(f[1]), int(f[2]), int(f[3]), float(f[4])))
    return key, rows


@pytest.mark.gpu
def test_large_chain_lattice_closed_form(klu, engine, tmp_path):
    K = 40
    assert max(unpruned_frontier(K)) > 2 ** 24  # the lattice the uncut frontier rejects
    p = chain_probs(K, 7)
    lat = chain_lattice(klu, "chain40", p)
    engine.load(klu.LatticeBatch.from_lattices([lat]))
    for nbest in (1, 100):
        want = closed_form_rows(p, nbest)
        got = engine.char_position([WS], nbest=nbest)[0]
        assert_rows_match(got, want, 2, what="chain position nbest %d" % nbest)
        assert [r[:4] for r in got] == [r[:4] for r in want]
        want = closed_form_rows(p, nbest, segment=True)
        got = engine.char_segment([WS], nbest=nbest)[0]
        assert_rows_match(got, want, 3, what="chain segment nbest %d" % nbest)
        assert [r[:3] for r in got] == [r[:3] for r in want]
    # the drop-in binary on the same lattice as a text archive (default --nbest 100)
    ark = str(tmp_path / "chain40.ark.txt")
    write_text_ark(ark, "chain40", K, p)
    assert len(klu.read_text_ark(ark)[0].src) == 3 * K
    tool = os.path.join(ROOT, "kaldi-lattice-utils_b200", "bin", "lattice-char-index-position")
    r = subprocess.run([tool, str(WS), "ark:" + ark, "ark,t:-"], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    key, got = parse_char_ark(r.stdout.decode())
    assert key == "chain40"
    want = engine.char_position([WS], nbest=100)[0]
    assert [x[:4] for x in got] == [x[:4] for x in want]
    assert max(abs(a[4] - b[4]) for a, b in zip(got, want)) <= TOL


# ---- oracle parity on lattices where the cut is active ------------------------------------
C5_LATTICES = 32


@pytest.fixture(scope="module")
def c5_batch(klu):
    return klu.synth_batch("c5", C5_LATTICES, seed=2024)


@pytest.fixture(scope="module")
def c5_oracle(ora, c5_batch):
    """The oracle's 100 best rows of every lattice, per (tool, groups); the n best for a smaller n
    are their first n (the oracle runs on host threads: a c5 lattice takes it seconds)."""
    from concurrent.futures import ThreadPoolExecutor
    lats = c5_batch.lattices()
    out = {}
    with ThreadPoolExecutor(max_workers=max(1, min(C5_LATTICES, os.cpu_count() or 1))) as ex:
        for tool in ("position", "segment"):
            fn = ora.char_position if tool == "position" else ora.char_segment
            for groups in GROUPS:
                out[tool, groups] = list(ex.map(lambda lat: fn(lat, [WS], other_groups=groups, nbest=100), lats))
    return out


GROUPS = [(), ((40,), (41,))]


@pytest.mark.gpu
@pytest.mark.parametrize("nbest", [1, 7, 100])
@pytest.mark.parametrize("groups", GROUPS)
def test_c5_cut_parity_position(engine, c5_batch, c5_oracle, nbest, groups):
    engine.load(c5_batch)
    got = engine.char_position([WS], other_groups=groups, nbest=nbest)
    for l in range(C5_LATTICES):
        want = c5_oracle["position", groups][l][:nbest]
        assert len(got[l]) == len(want)
        assert_rows_match(got[l], want, 2, what="c5 lat %d nbest %d groups %r" % (l, nbest, groups))


def _check_seg(got, want, what):
    # as test_gpu_char.py: rows as sorted multisets, keys exact, values within TOL, best first
    assert len(got) == len(want), what
    for g, w in zip(sorted(got, key=lambda r: (r[:3], -r[3])), sorted(want, key=lambda r: (r[:3], -r[3]))):
        assert g[:3] == w[:3], what
        assert abs(g[3] - w[3]) <= TOL, what
    for a, b in zip(got[:-1], got[1:]):
        assert a[3] >= b[3]


@pytest.mark.gpu
@pytest.mark.parametrize("nbest", [1, 7, 100])
@pytest.mark.parametrize("groups", GROUPS)
def test_c5_cut_parity_segment(engine, c5_batch, c5_oracle, nbest, groups):
    engine.load(c5_batch)
    got = engine.char_segment([WS], other_groups=groups, nbest=nbest)
    for l in range(C5_LATTICES):
        want = c5_oracle["segment", groups][l][:nbest]
        _check_seg(got[l], want, "c5 seg lat %d nbest %d groups %r" % (l, nbest, groups))


# ---- exact ties at the cut ----------------------------------------------------------------
def tie_lattice(klu, K):
    # both characters of a frame cost the same (dyadic costs: every sum is exact), so all the
    # strings of one (position, start, end) score exactly alike
    arcs = []
    for t in range(K):
        c = 0.5 + 0.25 * (t % 3)
        arcs += [(t, t + 1, 2 + 2 * t, c, 0.0, 1), (t, t + 1, 3 + 2 * t, c, 0.0, 1), (t, t + 1, WS, 1.0, 0.0, 1)]
    return klu.make_lattice("ties", K + 1, arcs, {K: (0.0, 0.0)})


@pytest.mark.gpu
@pytest.mark.parametrize("tool", ["position", "segment"])
def test_ties_at_the_cut(klu, engine, tool):
    K = 10
    engine.load(klu.LatticeBatch.from_lattices([tie_lattice(klu, K)]))
    run = engine.char_position if tool == "position" else engine.char_segment
    full = run([WS], nbest=100000)[0]
    assert len(full) < 100000  # tau stays -inf: nothing is cut
    lp = [r[-1] for r in full]
    # a cut inside a run of equal scores, deep enough that the frontier is cut before it
    n = next(i for i in range(40, len(lp) - 1) if lp[i - 1] == lp[i] and lp[i] != lp[0])
    cut_value = lp[n - 1]
    got = run([WS], nbest=n)[0]
    assert len(got) == n
    full_set = {r[:-1]: r[-1] for r in full}
    above = {r[:-1] for r in full if r[-1] > cut_value}
    got_keys = {r[:-1] for r in got}
    assert above <= got_keys
    for r in got:
        assert full_set[r[:-1]] == r[-1]
        assert r[:-1] in above or r[-1] == cut_value
