"""Generates tests/golden/*.npz from the reference's OWN code (oracle/_ref/libpxref.so =
pixsfm/base/src/cubic_hermite_spline_simd.h + pixsfm/base/src/graph.cc compiled verbatim by
oracle/Makefile from a reference checkout, REF=<path>).  Needs that library:
    python tests/golden/make_golden.py [spline graph spline_live]
(no argument: all fixtures).  The fixtures pin the oracle's restatement (tests/test_oracle_golden.py)
wherever the reference checkout is absent."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "pixel-perfect-sfm_b200"))
import oracle_lib as O  # noqa: E402

ref = O.ref()
assert ref is not None, "oracle/_ref/libpxref.so missing: run `make -C oracle`"
p = O.p


def spline_fixture():
    rng = np.random.default_rng(20260922)
    out = {}
    for name, dt, fn in (("f16", np.float16, ref.ref_spline_f16), ("f32", np.float32, ref.ref_spline_f32),
                         ("f64", np.float64, ref.ref_spline_f64)):
        C_ = 128
        n = 64
        P = rng.uniform(-1, 1, (n, 4, C_)).astype(dt)
        xs = np.concatenate([rng.uniform(0, 1, n - 4), [0.0, 0.5, 0.999999, 1e-9]])
        F = np.zeros((n, C_)); D = np.zeros((n, C_))
        for i in range(n):
            rc = fn(C_, p(P[i, 0]), p(P[i, 1]), p(P[i, 2]), p(P[i, 3]), C.c_double(xs[i]), p(F[i]), p(D[i]))
            assert rc == 0
        out["P_" + name] = P; out["x_" + name] = xs; out["f_" + name] = F; out["d_" + name] = D
    np.savez_compressed(os.path.join(HERE, "spline_ref.npz"), **out)


def graph_fixture():
    rng = np.random.default_rng(7)
    out = {}
    for g in range(6):
        n_img = int(rng.integers(3, 8)); per = int(rng.integers(5, 40))
        node_image = np.repeat(np.arange(n_img, dtype=np.int32), per)
        node_feature = np.tile(np.arange(per, dtype=np.int32), n_img)
        n = len(node_image)
        m = int(rng.integers(n, 4 * n))
        es = rng.integers(0, n, m).astype(np.int64); ed = rng.integers(0, n, m).astype(np.int64)
        keep = node_image[es] != node_image[ed]
        es, ed = es[keep], ed[keep]
        # quantised similarities force ties (exercises the (sim,node1,node2) tuple ordering)
        sim = np.round(rng.uniform(0.2, 1.0, len(es)), 1 if g % 2 == 0 else 6)
        # graph.cc iterates node by node over out_matches -> sort edges by source (stable)
        order = np.argsort(es, kind="stable")
        es, ed, sim = es[order], ed[order], sim[order]
        tl = np.zeros(n, np.int64); sc = np.zeros(n); rt = np.zeros(n, np.uint8)
        ref.ref_graph_labels(C.c_int64(n), p(node_image), p(node_feature), C.c_int64(len(es)), p(es), p(ed), p(sim),
                             p(tl), p(sc), p(rt))
        for k, v in dict(node_image=node_image, es=es, ed=ed, sim=sim, track_labels=tl, scores=sc, is_root=rt).items():
            out["g%d_%s" % (g, k)] = v
    out["n_graphs"] = np.array(6)
    np.savez_compressed(os.path.join(HERE, "graph_ref.npz"), **out)


def spline_live_fixture():
    """the input of test_live_reference_library_if_present and the reference's answer on it"""
    rng = np.random.default_rng(99)
    P = rng.uniform(-1, 1, (4, 4, 128)).astype(np.float16)
    x = rng.uniform(0, 1, 4)
    F = np.zeros((4, 128)); D = np.zeros((4, 128))
    for i in range(4):
        rc = ref.ref_spline_f16(128, p(P[i, 0]), p(P[i, 1]), p(P[i, 2]), p(P[i, 3]), C.c_double(x[i]), p(F[i]), p(D[i]))
        assert rc == 0
    np.savez_compressed(os.path.join(HERE, "spline_live_ref.npz"), P=P, x=x, f=F, d=D)


if __name__ == "__main__":
    fixtures = {"spline": spline_fixture, "graph": graph_fixture, "spline_live": spline_live_fixture}
    for name in sys.argv[1:] or fixtures:
        fixtures[name]()
    print("wrote", os.listdir(HERE))
