"""Pins the ORACLE: Philox known-answer vectors (Random123 kat_vectors) and the hand-derived known
answers of SURVEY.md A.8 (the reference itself ships no tests or golden files)."""
import hashlib
import json
import os

import numpy as np
import pytest

from helpers import GOLDEN
from oracle import philox as px
from oracle import sampler as sp
from oracle.em_read import bn_sort, em_read


def test_philox4x32_10_known_answers():
    kat = [
        ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
        ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
        ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
         (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
    ]
    for ctr, key, want in kat:
        got = px.philox4x32_10(np.array(ctr, dtype=np.uint32), key)
        assert tuple(int(v) for v in got) == want


def test_uniform_map_is_open_interval_and_exact():
    assert px.u01(0) == 2.0 ** -33 and px.u01(0xFFFFFFFF) == 1.0 - 2.0 ** -33
    ks = np.array([0, 1, 12345, 0xFFFFFFFF], dtype=np.uint32)
    assert np.all((px.u01(ks) * 2.0 ** 33) % 2 == 1)  # (2k+1) * 2^-33 exactly


def test_gate_threshold_matches_literal_comparison():
    for rate in [0.0127706, 0.5, 0.0547457, 1e-12, 2.0 ** -32, 2.0 ** -33, 0.999999, 1.0, 2.0, 0.0, -1.0, 0.126597]:
        G = px.gate_threshold(rate)
        if rate <= 0:
            assert G == 0
            continue
        if G > 0:
            assert px.u01(G - 1) < rate
        if G < 2 ** 32:
            assert not (px.u01(G) < rate)


def test_select_random_known_answers_balloon(model_paths):
    p = em_read(model_paths["balloon_v1"])
    w = p.N_initial[0][:, 0]
    assert w.tolist() == [28313, 5586, 2376, 0]
    for u, want in [(0.78, 1), (0.79, 2), (0.93, 2), (0.94, 3), (0.999999, 3)]:
        assert sp.select_random_u(w, u) == want
    w = p.N_initial[1][:, 1]
    assert w.tolist() == [526, 778, 531, 801, 2181, 651, 118]
    for u, want in [(0.1, 2), (0.5, 5), (0.9, 6)]:
        assert sp.select_random_u(w, u) == want
    # column-major layout: column sums of dh|L equal N{L}
    assert p.N_initial[1].sum(axis=0).tolist() == [28313, 5586, 2376, 0]
    assert p.zero_bins == [[], [4]]


def test_known_answers_uncor_v2p1(model_paths):
    p = em_read(model_paths["uncor_1200code_v2p1"])
    j = sp.asub2ind([4, 4, 4], [1, 4, 2])
    assert j == 29
    w = p.N_initial[3][:, j - 1]
    assert w.tolist() == [443463, 4990916, 44740943, 97447270, 37004039, 21079156, 8113940, 329967]
    assert w.sum() == 214149694 == p.N_initial[2][1, 12]
    for u, want in [(0.05, 3), (0.5, 4), (0.95, 6)]:
        assert sp.select_random_u(w, u) == want
    # transition columns for (A=4,L=2,v=4,dv=3,dh=4,dpsi=4)
    x = np.array([1, 4, 2, 4, 3, 4, 4, 0, 0, 0], dtype=float)
    G, r = p.G_transition, p.r_transition
    js = [sp.asub2ind(r[G[:, i]], x[G[:, i]]) for i in (7, 8, 9)]
    assert js == [3918, 1960, 558]
    assert p.N_transition[7][:, js[0] - 1].tolist() == [0, 60988, 72970079, 25979, 0]
    assert p.N_transition[8][:, js[1] - 1].tolist() == [0, 1, 329077, 146303227, 172254, 0, 0]
    assert p.N_transition[9][:, js[2] - 1].tolist() == [0, 0, 111876, 89789351, 97929, 0, 0]
    assert p.zero_bins == [[], [], [], [], [3], [4], [4]]            # UncorEncounterModel.m:84
    assert sp.dediscretize_u(2, p.boundaries[2], p.zero_bins[2], lambda: 0.25) == 1650.0
    assert sp.dediscretize_u(4, p.boundaries[5], p.zero_bins[5], lambda: 0.9) == 0.0
    assert sp.dediscretize_u(3, p.boundaries[0], p.zero_bins[0], lambda: 0.9) == 3


def test_all_zero_column_selects_bin_one():
    assert sp.select_random_u(np.zeros(5), 0.73) == 1
    assert sp.select_random_u(np.array([0, 0, 3.0, 0]), 1e-9) == 3   # leading zero-weight bins are skipped


def test_bn_sort_orders(model_paths):
    assert em_read(model_paths["paramotor_v1"]).order_initial == [1, 2, 5, 4, 3]
    assert em_read(model_paths["glider_v1"]).order_transition == [1, 2, 3, 4, 5, 7, 8, 6]
    assert em_read(model_paths["cor_v1"]).order_initial == [2, 1, 5, 6, 11, 12, 8, 7, 4, 9, 10, 13, 14, 16, 15, 3]
    with pytest.raises(Exception, match="hierarchically sorted"):
        bn_sort(np.array([[0, 1], [1, 0]], dtype=bool))


def test_events_expansion_semantics():
    # events2samples.m / events2controls.m on a hand-made list: [dt var value]
    initial = np.array([10.0, 20.0])
    events = [[2, 1, 11.0], [0, 2, 21.0], [3, 2, 22.0], [1, 0, 0]]
    d = sp.events2samples(initial, events)
    assert d.shape == (2, 6)
    assert d[0].tolist() == [10, 10, 11, 11, 11, 11]
    assert d[1].tolist() == [20, 20, 21, 21, 21, 22]
    c = sp.events2controls(initial, events, np.array([[2, 3]]))
    assert c.tolist() == [[0, 20], [2, 21], [5, 22]]


def test_preset_dependent_variable_errors(model_paths):
    from oracle.uniforms import KeyedPhilox
    p = em_read(model_paths["uncor_1200code_v2p1"])
    U = KeyedPhilox(1).bind(p.n_initial, p.temporal_map, p.resample_rates)
    a = sp.bn_dirichlet_prior(p.N_initial, 0)
    with pytest.raises(sp.OracleError, match="Attempt to preset a dependent variable"):
        sp.bn_sample(p.G_initial, p.r_initial, p.N_initial, a, 1, [None, 2] + [None] * 5, p.order_initial, U)


def parsed_tables_digest(p):
    """sha256 of what em_read parses from a model file: labels, G_initial, every N table, boundaries, resample_rates."""
    h = hashlib.sha256()
    for labels in (p.labels_initial, p.labels_transition or []):
        h.update("\n".join(labels).encode() + b"\0")
    for x in [p.G_initial] + list(p.N_initial) + list(p.N_transition or []) + list(p.boundaries) + [p.resample_rates]:
        if x is None:
            h.update(b"-")
        else:
            a = np.ascontiguousarray(x, dtype="<f8")
            h.update(repr(a.shape).encode() + a.tobytes())
    return h.hexdigest()


def test_fixture_archive_matches_reference_files(model_paths):
    """The archived models parse to the same tables as the upstream model/*.txt files they were packed from
    (tests/golden/upstream_reference.json: model_digests)."""
    want = json.load(open(os.path.join(GOLDEN, "upstream_reference.json")))["model_digests"]
    assert sorted(want) == sorted(model_paths)
    for name, path in model_paths.items():
        assert parsed_tables_digest(em_read(path)) == want[name], name


def test_spec_v3_word_bijections_equidistribute():
    """Stream spec v3 (oracle/philox.py): select on k, gate on k*A, de-discretisation on k*B.  Over any interval of
    words (= any bin of a select) the gate must fire at its rate and u_dd must be uniform, also given the gate."""
    from oracle import philox as px
    rs = np.random.RandomState(3)
    A, B, M = np.uint64(px.GATE_MULT), np.uint64(px.DD_MULT), np.uint64(0xFFFFFFFF)
    assert px.GATE_MULT % 2 == 1 and px.DD_MULT % 2 == 1            # bijections of the 32-bit words
    for L_ in (20_000, 1_000_000):
        for rate in (0.0107, 0.0333, 0.6667):
            lo = rs.randint(0, 2 ** 32 - L_)
            k = (np.uint64(lo) + np.arange(L_, dtype=np.uint64)) & M
            fired = ((k * A) & M) < np.uint64(px.gate_threshold(rate))
            assert abs(fired.mean() - rate) < 4.0 / L_ + 1e-4 * rate      # low-discrepancy lattice, far better than binomial
            u = (((k * B) & M) >> np.uint64(9)).astype(np.float64) * 2.0 ** -23
            for sub in (u, u[fired]):
                h = np.histogram(sub, bins=16, range=(0, 1))[0]
                assert np.abs(h - sub.size / 16).max() < 0.02 * sub.size / 16 + 12
    k = int(rs.randint(0, 2 ** 32))
    assert px.dd_uniform(k) == ((((k * px.DD_MULT) & 0xFFFFFFFF) >> 9) + 0.5) * 2.0 ** -23
    assert 0.0 < px.dd_uniform(0) < 1.0 and 0.0 < px.dd_uniform(0xFFFFFFFF) < 1.0
