"""lattice-char-index-utterance in the CPU reference (tests/char_utterance_ref.cc): the first-occurrence
DP (CharIndexUtterance) against the definition applied to the list of all paths (BruteCharUtterance)."""
import math
import os

import numpy as np
import pytest

import char_utterance_ref as ref
from test_gpu_char_prune import chain_lattice, chain_probs, closed_form_rows
from util import GOLD, assert_rows_match, char_lattice

WS = 1
FLAGS = [dict(), dict(acoustic_scale=0.5), dict(graph_scale=0.8, insertion_penalty=0.3), dict(beam=4.0)]
GROUPS = [(), ((40,), (41,))]


def _lattices(klu):
    rng = np.random.RandomState(77)
    lats = [char_lattice(klu, rng, "c%d" % i, nwords=int(rng.randint(1, 4)), punct=(40, 41),
                         eps_prob=0.1 if i % 2 else 0.0) for i in range(16)]
    lats.append(repeat_lattice(klu))
    return lats


def repeat_lattice(klu):
    """'2' can occur twice on one path: 2 ws 2, 2 ws 3, 3 ws 2 (and an epsilon detour)."""
    arcs = [(0, 1, 2, 0.3, 0.2, 1), (0, 1, 3, 1.1, 0.4, 1), (1, 2, WS, 0.2, 0.0, 1), (1, 2, 0, 1.5, 0.0, 1),
            (2, 3, 2, 0.7, 0.1, 1), (2, 3, 3, 0.9, 0.3, 1)]
    return klu.make_lattice("rep", 4, arcs, {3: (0.0, 0.0)})


def _position_sums(ora, lat, wspace=(WS,)):
    s = {}
    for r in ora.char_position(lat, list(wspace), nbest=10 ** 9):
        s[r[0]] = np.logaddexp(s.get(r[0], -np.inf), r[-1])
    return s


@pytest.mark.parametrize("flags", FLAGS)
@pytest.mark.parametrize("groups", GROUPS)
def test_dp_matches_brute_force(klu, flags, groups):
    for lat in _lattices(klu):
        full = ref.char_utterance(lat, [WS], other_groups=groups, nbest=10 ** 9, **flags)
        brute = ref.brute_char_utterance(lat, [WS], other_groups=groups, nbest=10 ** 9, **flags)
        assert_rows_match(full, brute, 1, what="%s %r %r" % (lat.key, flags, groups))
        for nbest in (1, 3):
            got = ref.char_utterance(lat, [WS], other_groups=groups, nbest=nbest, **flags)
            assert got == full[:nbest]
            want = brute[:nbest]
            assert len(got) == len(want)
            for g, w in zip(got, want):
                assert abs(g[1] - w[1]) <= 1e-9
                assert g[0] == w[0] or abs(g[1] - w[1]) <= 1e-9


def test_readme_char_lattice(klu, ora):
    lat = klu.read_text_ark(os.path.join(GOLD, "lattice.char.ark.txt"))[0]
    got = ref.char_utterance(lat, [28])
    assert_rows_match(got, ref.brute_char_utterance(lat, [28]), 1)
    assert len(got) == 8
    # '20_8_5' occurs twice on every path: probability one, below its expected count
    assert dict(got)["20_8_5"] == pytest.approx(0.0, abs=1e-9)
    assert _position_sums(ora, lat, [28])["20_8_5"] > 0.1


def test_probability_not_expected_count(klu, ora):
    lat = repeat_lattice(klu)
    got = dict(ref.char_utterance(lat, [WS], nbest=10 ** 9))
    sums = _position_sums(ora, lat)
    assert set(got) == set(sums)
    assert got["2"] < sums["2"] - 1e-3  # two occurrences on one path count once
    assert got["3"] < sums["3"] - 1e-3
    for lat in [chain_lattice(klu, "chain", chain_probs(6, seed)) for seed in (1, 2)]:
        got = dict(ref.char_utterance(lat, [WS], nbest=10 ** 9))
        sums = _position_sums(ora, lat)
        assert set(got) == set(sums)
        for k, v in got.items():  # labels are private to a frame: no string repeats on a path
            assert v == pytest.approx(sums[k], abs=1e-12)


def test_chain_closed_form_small(klu):
    for seed in (1, 2):
        p = chain_probs(7, seed)
        lat = chain_lattice(klu, "small", p)
        for nbest in (1, 5, 100000):
            want = [(r[0], r[-1]) for r in closed_form_rows(p, nbest, segment=True)]
            got = ref.char_utterance(lat, [WS], nbest=nbest)
            assert_rows_match(got, want, 1, what="closed form nbest %d" % nbest)
            assert len(got) == len(want)
            assert all(not math.isnan(v) for _, v in got)
