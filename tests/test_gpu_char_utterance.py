"""lattice-char-index-utterance on the GPU (klu_char.cu, k_char_occ) against the CPU reference
(tests/char_utterance_ref.cc), a closed form at scale, the n-best cut, exact ties and the drop-in binary."""
import os
import struct
import subprocess

import numpy as np
import pytest

import char_utterance_ref as ref
from test_gpu_char_prune import chain_lattice, chain_probs, closed_form_rows, unpruned_frontier, write_text_ark
from util import GOLD, TOL, assert_rows_match, char_lattice

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "kaldi-lattice-utils_b200", "bin", "lattice-char-index-utterance")
WS = 1
CASES = [dict(), dict(acoustic_scale=0.5), dict(graph_scale=0.8, insertion_penalty=0.3), dict(beam=4.0),
         dict(nbest=7), dict(nbest=100000)]
GROUPS = [(), ((40,), (41,))]
C5_LATTICES = 32


def _check(got, want, what):
    assert len(got) == len(want), what
    assert_rows_match(got, want, 1, what=what)


@pytest.mark.parametrize("flags", CASES)
def test_parity_random(klu, engine, flags):
    rng = np.random.RandomState(1234)
    lats = [char_lattice(klu, rng, "c%d" % i, nwords=int(rng.randint(1, 5))) for i in range(12)]
    lats.insert(4, klu.make_lattice("empty", 0, [], {}))
    engine.load(klu.LatticeBatch.from_lattices(lats))
    got = engine.char_utterance([WS], **flags)
    for l, lat in enumerate(lats):
        _check(got[l], ref.char_utterance(lat, [WS], **flags), "lat %d %r" % (l, flags))


def test_parity_other_groups_and_epsilons(klu, engine):
    rng = np.random.RandomState(99)
    lats = [char_lattice(klu, rng, "p%d" % i, nwords=3, punct=(40, 41), eps_prob=0.1) for i in range(8)]
    engine.load(klu.LatticeBatch.from_lattices(lats))
    got = engine.char_utterance([WS], other_groups=[[40], [41]], nbest=100000)
    for l, lat in enumerate(lats):
        _check(got[l], ref.char_utterance(lat, [WS], other_groups=[[40], [41]], nbest=100000), "punct lat %d" % l)


def test_readme_char_lattice(klu, engine):
    lat = klu.read_text_ark(os.path.join(GOLD, "lattice.char.ark.txt"))[0]
    engine.load(klu.LatticeBatch.from_lattices([lat]))
    _check(engine.char_utterance([28])[0], ref.char_utterance(lat, [28]), "README char lattice")


@pytest.fixture(scope="module")
def c5_batch(klu):
    return klu.synth_batch("c5", C5_LATTICES, seed=2024)


@pytest.fixture(scope="module")
def c5_ref(c5_batch):
    from concurrent.futures import ThreadPoolExecutor
    lats = c5_batch.lattices()
    out = {}
    with ThreadPoolExecutor(max_workers=max(1, min(C5_LATTICES, os.cpu_count() or 1))) as ex:
        for groups in GROUPS:
            out[groups] = list(ex.map(lambda lat: ref.char_utterance(lat, [WS], other_groups=groups, nbest=100), lats))
    return out


@pytest.mark.parametrize("nbest", [1, 7, 100])
@pytest.mark.parametrize("groups", GROUPS)
def test_c5_parity(engine, c5_batch, c5_ref, nbest, groups):
    engine.load(c5_batch)
    got = engine.char_utterance([WS], other_groups=groups, nbest=nbest)
    for l in range(C5_LATTICES):
        _check(got[l], c5_ref[groups][l][:nbest], "c5 lat %d nbest %d groups %r" % (l, nbest, groups))


def test_c5_cut_never_changes_a_result(engine, c5_batch):
    engine.load(c5_batch)
    full = engine.char_utterance([WS], nbest=100)
    for k in (1, 7, 50):
        got = engine.char_utterance([WS], nbest=k)
        for l in range(C5_LATTICES):
            assert got[l] == full[l][:k], "c5 lat %d nbest %d" % (l, k)


def _utt_closed_form(p, nbest):
    return [(r[0], r[-1]) for r in closed_form_rows(p, nbest, segment=True)]


def test_chain_closed_form_reference_small(klu):
    for seed in (1, 2):
        p = chain_probs(7, seed)
        lat = chain_lattice(klu, "small", p)
        for nbest in (1, 5, 100000):
            got = ref.char_utterance(lat, [WS], nbest=nbest)
            _check(got, _utt_closed_form(p, nbest), "reference closed form nbest %d" % nbest)


def parse_text(text):
    out = []
    for line in text.strip().split("\n"):
        key, rest = (line.split(" ", 1) + [""])[:2]
        rows = []
        for ent in rest.split(";"):
            f = ent.split()
            if f:
                rows.append((f[0], float(f[1])))
        out.append((key, rows))
    return out


def parse_binary(b):
    out = []
    p = 0
    while p < len(b):
        sp = b.index(b" ", p)
        key = b[p:sp].decode()
        p = sp + 1
        assert b[p:p + 2] == b"\0B" and b[p + 2] == 4
        n = struct.unpack("<i", b[p + 3:p + 7])[0]
        p += 7
        rows = []
        for _ in range(n):
            sp = b.index(b" ", p)
            s = b[p:sp].decode()
            p = sp + 1
            assert b[p] == 8
            rows.append((s, struct.unpack("<d", b[p + 1:p + 9])[0]))
            p += 9
        out.append((key, rows))
    return out


def test_large_chain_closed_form(klu, engine, tmp_path):
    K = 40
    assert max(unpruned_frontier(K)) > 2 ** 24  # the uncut frontier of the position keys; strings alone are fewer
    p = chain_probs(K, 7)
    lat = chain_lattice(klu, "chain40", p)
    engine.load(klu.LatticeBatch.from_lattices([lat]))
    for nbest in (1, 100):
        want = _utt_closed_form(p, nbest)
        got = engine.char_utterance([WS], nbest=nbest)[0]
        _check(got, want, "chain nbest %d" % nbest)
        assert [r[0] for r in got] == [r[0] for r in want]
    ark = str(tmp_path / "chain40.ark.txt")
    write_text_ark(ark, "chain40", K, p)
    for nbest in (1, 100):
        r = subprocess.run([TOOL, "--nbest=%d" % nbest, str(WS), "ark:" + ark, "ark,t:-"], capture_output=True)
        assert r.returncode == 0, r.stderr.decode()
        [(key, got)] = parse_text(r.stdout.decode())
        assert key == "chain40"
        want = _utt_closed_form(p, nbest)
        assert [x[0] for x in got] == [x[0] for x in want]
        assert max(abs(a[1] - b[1]) for a, b in zip(got, want)) <= TOL


def mirror_lattice(klu, tail=True):
    """Two mirrored branches: '2_3' and '4_5' have the same arcs, costs and exits (dyadic costs);
    with the tail, '7' (more probable) and '6' (less) follow them."""
    arcs = [(0, 1, 2, 0.5, 0.25, 1), (0, 3, 4, 0.5, 0.25, 1), (1, 2, 3, 0.75, 0.0, 1), (3, 4, 5, 0.75, 0.0, 1),
            (2, 5, WS, 0.25, 0.0, 1), (4, 5, WS, 0.25, 0.0, 1)]
    if not tail:
        return klu.make_lattice("mirror", 6, arcs, {5: (0.0, 0.0)})
    arcs += [(5, 6, 6, 1.0, 0.0, 1), (5, 6, 7, 0.5, 0.0, 1)]
    return klu.make_lattice("mirror", 7, arcs, {6: (0.0, 0.0)})


@pytest.mark.parametrize("tail", [False, True])
def test_ties_go_to_the_smaller_string(klu, engine, tail):
    lat = mirror_lattice(klu, tail)
    engine.load(klu.LatticeBatch.from_lattices([lat]))
    full = engine.char_utterance([WS], nbest=100)[0]
    _check(full, ref.char_utterance(lat, [WS], nbest=100), "mirror")
    val = dict(full)
    assert val["2_3"] == val["4_5"]  # bit-identical occurrence DPs
    if tail:  # '7', then the tied pair: a cut after two rows falls inside the tie
        assert val["7"] > val["2_3"] > val["6"]
        assert [r[0] for r in engine.char_utterance([WS], nbest=2)[0]] == ["7", "2_3"]
    else:
        assert [r[0] for r in full] == ["2_3", "4_5"]
        assert [r[0] for r in engine.char_utterance([WS], nbest=1)[0]] == ["2_3"]


def test_cli_text_and_binary_match_engine(klu, engine, tmp_path):
    ark = str(tmp_path / "c5.ark.txt")
    cfg = klu.lattice.SHAPES["c5"]
    subprocess.run([os.path.join(ROOT, "kaldi-lattice-utils_b200", "bin", "klu-synth-lattices")] + [str(cfg[k]) for k in (
        "frames", "states_per_frame", "arcs_per_state", "max_skip", "vocab", "pool_size", "window", "eps_prob",
        "weight_max", "kind")] + ["5", "6", "ark,t:" + ark], check=True)
    lats = klu.read_text_ark(ark)
    engine.load(klu.LatticeBatch.from_lattices(lats))
    want = engine.char_utterance([WS], nbest=20)
    r = subprocess.run([TOOL, "--nbest=20", str(WS), "ark:" + ark, "ark,t:-"], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    text = parse_text(r.stdout.decode())
    assert [k for k, _ in text] == [lat.key for lat in lats]
    out = tmp_path / "out.ark"
    r = subprocess.run([TOOL, "--nbest=20", str(WS), "ark:" + ark, "ark:" + str(out)], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    binary = parse_binary(out.read_bytes())
    assert [k for k, _ in binary] == [lat.key for lat in lats]
    for l in range(len(lats)):
        assert len(want[l]) == 20
        assert [x[0] for x in binary[l][1]] == [x[0] for x in want[l]]
        assert [x[1] for x in binary[l][1]] == [x[1] for x in want[l]]  # doubles, bit for bit
        assert [x[0] for x in text[l][1]] == [x[0] for x in want[l]]
        assert all(abs(a[1] - b[1]) <= 1e-6 * max(1.0, abs(b[1])) for a, b in zip(text[l][1], want[l]))


def test_cli_error_exit_code(tmp_path):
    bad = tmp_path / "bad.txt"
    bad.write_text("cyc\n0 1 2 0,0,1\n1 0 3 0,0,1\n1\n\n")
    r = subprocess.run([TOOL, str(WS), "ark:" + str(bad), "ark,t:-"], capture_output=True)
    assert r.returncode == 1 and b"cyclic" in r.stderr
