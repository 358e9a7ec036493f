"""Oracle vs fixtures generated FROM THE REFERENCE'S OWN CODE (tests/golden/make_golden.py):
the AVX2 spline header and graph.cc compiled verbatim.  Bit-exact.  Also checks the live
oracle/_ref library when it is present."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
p = O.p


def _oracle_spline(name, P, x):
    L = O.lib()
    n, _, C_ = P.shape
    F = np.zeros((n, C_)); D = np.zeros((n, C_))
    for i in range(n):
        for ch in range(C_):
            taps = np.ascontiguousarray(P[i, :, ch])
            if name == "f64":
                f = C.c_double(); d = C.c_double()
                L.orc_spline_f64(p(taps), C.c_double(x[i]), C.byref(f), C.byref(d))
            else:
                f = C.c_float(); d = C.c_float()
                getattr(L, "orc_spline_" + name)(p(taps), C.c_double(x[i]), C.byref(f), C.byref(d))
            F[i, ch] = f.value; D[i, ch] = d.value
    return F, D


@pytest.mark.parametrize("name", ["f16", "f32", "f64"])
def test_spline_bit_exact_vs_reference_header(name):
    z = np.load(os.path.join(GOLD, "spline_ref.npz"))
    P, x = z["P_" + name], z["x_" + name]
    F, D = _oracle_spline(name, P[:24], x[:24])
    assert np.array_equal(F, z["f_" + name][:24])
    assert np.array_equal(D, z["d_" + name][:24])


def test_graph_labels_bit_exact_vs_reference_graph_cc():
    z = np.load(os.path.join(GOLD, "graph_ref.npz"))
    L = O.lib()
    for g in range(int(z["n_graphs"])):
        ni = z["g%d_node_image" % g]; es = z["g%d_es" % g]; ed = z["g%d_ed" % g]; sim = z["g%d_sim" % g]
        n = len(ni)
        tl = np.zeros(n, np.int64); sc = np.zeros(n); rt = np.zeros(n, np.uint8)
        L.orc_graph_track_labels(C.c_int64(n), p(ni), C.c_int64(len(es)), p(es), p(ed), p(sim), p(tl))
        L.orc_graph_score_labels(C.c_int64(n), C.c_int64(len(es)), p(es), p(ed), p(sim), p(tl), p(sc))
        L.orc_graph_root_labels(C.c_int64(n), p(tl), p(sc), p(rt))
        assert np.array_equal(tl, z["g%d_track_labels" % g])
        assert np.array_equal(sc, z["g%d_scores" % g])
        assert np.array_equal(rt, z["g%d_is_root" % g])
        # one-feature-per-image constraint inside every track
        for t in np.unique(tl):
            imgs = ni[tl == t]
            assert len(imgs) == len(np.unique(imgs))


def test_live_reference_library_if_present():
    """the oracle against the reference's answer stored in spline_live_ref.npz and, where oracle/_ref was built, against
    the live library on the same input"""
    z = np.load(os.path.join(GOLD, "spline_live_ref.npz"))
    P, x = z["P"], z["x"]
    F2, D2 = _oracle_spline("f16", P, x)
    assert np.array_equal(F2, z["f"]) and np.array_equal(D2, z["d"])
    ref = O.ref()
    if ref is None:
        return
    F = np.zeros((4, 128)); D = np.zeros((4, 128))
    for i in range(4):
        ref.ref_spline_f16(128, p(P[i, 0]), p(P[i, 1]), p(P[i, 2]), p(P[i, 3]), C.c_double(x[i]), p(F[i]), p(D[i]))
    assert np.array_equal(F, F2) and np.array_equal(D, D2)


def test_ka_problem_labels_first_fit_decreasing():
    # python restatement of keypoint_adjustment/main.py:13-57 (the reference IS python here)
    from collections import Counter
    import sys

    def ref_labels(track_labels, max_per_problem):
        track_count = Counter(track_labels)
        bins = []
        t2p = [-1] * len(track_count)
        start = 0; last_v = sys.maxsize
        for k, v in track_count.most_common():
            if v < last_v:
                start = 0; last_v = v
            found = False
            if v < max_per_problem:
                for i in range(start, len(bins)):
                    if bins[i] + v <= max_per_problem:
                        bins[i] += v; t2p[k] = i; found = True; start = i
                        break
            if not found:
                t2p[k] = len(bins); start = len(bins); bins.append(v)
        return [t2p[v] for v in track_labels], bins

    rng = np.random.default_rng(1)
    for trial in range(5):
        n_tracks = int(rng.integers(5, 200))
        sizes = rng.integers(1, 12, n_tracks)
        labels = np.repeat(np.arange(n_tracks), sizes)
        rng.shuffle(labels)
        # labels must be 0..n_tracks-1 (compute_track_labels numbering)
        exp, bins = ref_labels(labels.tolist(), 50 if trial else 10)
        out = np.zeros(len(labels), np.int32)
        nb = O.lib().orc_ka_problem_labels(C.c_int64(len(labels)), p(labels.astype(np.int64)), 50 if trial else 10, p(out))
        assert nb == len(bins)
        assert out.tolist() == exp
