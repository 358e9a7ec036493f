"""util/h5lite.py — the classic-layout HDF5 subset in pure Python.  Read side against REAL HDF5 files: the ten
h5py-written calibration files the reference ships with its sacre_coeur dataset (datasets/sacre_coeur/ground_truth/),
kept under tests/golden/calibration/.  Their content is self-checking: K is an intrinsics matrix, R a rotation, q the
same rotation as a unit quaternion.  Write side: round trips
(nested groups, many links, chunked patches, attributes), and the hloc / feature-cache helpers on top of it."""
import glob
import os

import numpy as np
import pytest

from pixsfm.util import h5lite, hloc

HERE = os.path.dirname(os.path.abspath(__file__))


def _quat_to_R(q):
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _check_calibration(path):
    f = h5lite.File(path)
    assert f.keys() == ["K", "R", "T", "q"]
    K, R, T, q = (np.asarray(f[k]) for k in ("K", "R", "T", "q"))
    assert K.shape == (3, 3) and K.dtype == np.float64 and R.shape == (3, 3) and T.shape == (3,) and q.shape == (4,)
    assert K[2, 2] == 1.0 and K[1, 0] == K[2, 0] == K[2, 1] == 0.0 and K[0, 0] > 100 and K[0, 0] == K[1, 1] and K[0, 2] > 0
    assert np.abs(R.T @ R - np.eye(3)).max() < 1e-12 and abs(np.linalg.det(R) - 1) < 1e-12
    assert abs(np.linalg.norm(q) - 1) < 1e-12 and np.abs(_quat_to_R(q) - R).max() < 1e-6


def test_reads_real_hdf5_files():
    paths = sorted(glob.glob(os.path.join(HERE, "golden", "calibration", "calibration_*.h5")))
    assert len(paths) == 10
    for path in paths:
        _check_calibration(path)


def test_round_trip_groups_datasets_attributes(tmp_path):
    rng = np.random.default_rng(0)
    path = tmp_path / "t.h5"
    patches = rng.normal(size=(7, 4, 4, 16)).astype(np.float16)
    with h5lite.File(path, "w") as f:
        f.attrs["version"] = 3
        g = f.create_group("mapping/image_0001.jpg")
        g.attrs["format"] = 2; g.attrs["is_sparse"] = 1; g.attrs["scale"] = np.array([1.0, 0.25]); g.attrs["name"] = "s2dnet"
        g.create_dataset("patches", data=patches, chunks=(1, 4, 4, 16))
        g.create_dataset("keypoint_ids", data=np.arange(7, dtype=np.int32))
        g.create_dataset("corners", data=rng.integers(0, 900, (7, 2)).astype(np.int32))
        for k in range(40):                       # more links than one default symbol node holds
            f.create_dataset("many/d%03d" % k, data=np.full((3,), k, np.float64))
        f.create_dataset("empty", data=np.zeros((0, 2), np.float32))
        f.create_dataset("scalar", data=np.float64(2.5))
    f = h5lite.File(path)
    assert f.attrs["version"] == 3 and set(f.keys()) == {"mapping", "many", "empty", "scalar"}
    g = f["mapping/image_0001.jpg"]
    assert g.attrs["format"] == 2 and g.attrs["name"] == "s2dnet" and np.array_equal(g.attrs["scale"], [1.0, 0.25])
    assert np.array_equal(np.asarray(g["patches"]), patches) and g["patches"].dtype == np.float16
    assert np.array_equal(g["patches"][3], patches[3]) and g["keypoint_ids"][6] == 6
    assert f["many"].keys() == ["d%03d" % k for k in range(40)] and f["many/d017"][1] == 17.0
    assert np.asarray(f["empty"]).shape == (0, 2) and np.asarray(f["scalar"]).shape == () and float(np.asarray(f["scalar"])) == 2.5
    assert "mapping/image_0001.jpg/patches" in f and "nope" not in f
    seen = []
    f.visititems(lambda name, obj: seen.append(name) if isinstance(obj, h5lite.Dataset) else None)
    assert "mapping/image_0001.jpg/patches" in seen and len(seen) == 3 + 40 + 2
    assert g["patches"].parent.name.strip("/") == "mapping/image_0001.jpg"


def test_hloc_files_through_h5lite(tmp_path):
    rng = np.random.default_rng(1)
    kp = {"db/a.jpg": rng.uniform(0, 100, (5, 2)), "q/b.jpg": rng.uniform(0, 100, (3, 2))}
    hloc.write_keypoints_hloc(tmp_path / "kp.h5", kp)
    got = hloc.read_keypoints_hloc(tmp_path / "kp.h5")
    assert set(got) == set(kp) and all(np.array_equal(got[k], kp[k]) for k in kp)
    assert hloc.list_h5_names(tmp_path / "kp.h5") == sorted(kp)
    # a match file as hloc writes it: group "<name0 with / -> ->/<name1 ...>", matches0 + matching_scores0
    with h5lite.File(tmp_path / "m.h5", "w") as f:
        g = f.create_group("db-a.jpg/q-b.jpg")
        g.create_dataset("matches0", data=np.array([-1, 2, 0, -1, 1], np.int64))
        g.create_dataset("matching_scores0", data=np.array([0, .9, .8, 0, .7], np.float32))
    (m,), (s,) = hloc.read_matches_hloc(tmp_path / "m.h5", [("db/a.jpg", "q/b.jpg")])
    assert m.tolist() == [[1, 2], [2, 0], [4, 1]] and np.allclose(s, [.9, .8, .7])
    (mr,), _ = hloc.read_matches_hloc(tmp_path / "m.h5", [("q/b.jpg", "db/a.jpg")])
    assert mr.tolist() == [[2, 1], [0, 2], [1, 4]]


@pytest.mark.parametrize("cache_format", ["chunked", "grouped"])
def test_feature_cache_round_trip(tmp_path, cache_format):
    """the dense-feature cache of extract.py:98-128 (both storage formats of featuremap.cc) -> FeatureManager"""
    from pixsfm import features
    from pixsfm.features import store_features
    rng = np.random.default_rng(2)
    fm = features.FeatureManager([16, 8], np.float16)
    for level, ch in enumerate((16, 8)):
        for name in ("a.jpg", "seq/b.jpg"):
            n = 5 + level
            fm.fset(level).emplace(name, features.FeatureMap(rng.normal(size=(n, 6, 6, ch)).astype(np.float16), [3 * k + 1 for k in range(n)],
                                                           rng.integers(0, 500, (n, 2)).astype(np.int32),
                                                           {"scale": (1.0 / (1 + level),) * 2, "is_sparse": True}))
    store_features.write_feature_manager_cache(tmp_path / "cache.h5", fm, cache_format)
    got = store_features.load_features_from_cache(tmp_path / "cache.h5")
    assert got.num_levels == 2
    for level in range(2):
        assert sorted(got.fset(level).keys()) == ["a.jpg", "seq/b.jpg"] and got.fset(level).channels == fm.fset(level).channels
        for name in ("a.jpg", "seq/b.jpg"):
            a, b = fm.fset(level).fmap(name), got.fset(level).fmap(name)
            assert a.point2D_ids == b.point2D_ids and np.array_equal(a.corners, b.corners) and np.array_equal(a.scale, b.scale)
            assert b.patches.dtype == np.float16 and np.array_equal(a.patches, b.patches) and b.is_sparse


def test_dense_map_stored_once_is_read_back_as_patches(tmp_path):
    """featuremap.cc:158-166: a dense map with several keypoint ids and a patch_size comes back as sparse patches cut at the corners"""
    from pixsfm.features import store_features
    rng = np.random.default_rng(3)
    dense = rng.normal(size=(1, 40, 50, 8)).astype(np.float16)
    corners = np.array([[3, 4], [20, 10], [34, 24]], np.int32)
    with h5lite.File(tmp_path / "d.h5", "w") as f:
        f.attrs["channels_per_level"] = [8]; f.attrs["dtype"] = "half"
        g = f.create_group("0/img.jpg")
        store_features.write_featuremap_cache(g, [7, 8, 9], dense, corners, np.ones((3, 2)), {"is_sparse": False, "patch_size": 16, "scale": np.ones(2)})
    fm = store_features.load_features_from_cache(tmp_path / "d.h5")
    m = fm.fset(0).fmap("img.jpg")
    assert m.is_sparse and m.point2D_ids == [7, 8, 9] and m.patches.shape == (3, 16, 16, 8)
    assert np.array_equal(m.patches[1], dense[0, 10:26, 20:36])


def test_lazy_cache_loads_per_feature_view_and_unloads(tmp_path):
    """FeatureManager(path, fill=False) (extract.py:218-222, featuremap.h:43-71): metadata is resident, the patches of an
    image arrive when a FeatureView covers it and leave with the view; the problem built from a lazily filled set is the
    one built from the in-memory set."""
    from pixsfm import features
    from pixsfm._pixsfm import _bundle_adjustment as ba
    from pixsfm._pixsfm._features import LazyFeatureMap
    from pixsfm.features import store_features
    from recon_util import make_reconstruction
    rec, fm, _, _ = make_reconstruction(n_cams=5, n_points=30, track_len=3, channels=16, seed=4)
    store_features.write_feature_manager_cache(tmp_path / "cache.h5", fm)
    lazy = store_features.load_features_from_cache(tmp_path / "cache.h5", fill=False)
    fset = lazy.fset(0)
    maps = [fset.fmap(n) for n in fset.keys()]
    assert len(maps) == 5 and all(isinstance(m, LazyFeatureMap) and not m.is_loaded for m in maps)
    ref = fm.fset(0)
    for name in ref.keys():                                   # metadata without a single patch read
        a, b = ref.fmap(name), fset.fmap(name)
        assert a.point2D_ids == b.point2D_ids and np.array_equal(a.corners, b.corners) and np.array_equal(a.scale, b.scale)
        assert b.shape == a.shape and b.channels == 16 and b.dtype == a.dtype and b.size() == a.size() and b.has_point2D(0)
    assert not any(m.is_loaded for m in maps)

    class Two:                                                # a view over two of the five images
        images = {i: rec.images[i] for i in (1, 2)}
    with features.FeatureView(fset, Two) as view:
        assert sorted(n for n in fset.keys() if fset.fmap(n).is_loaded) == ["image000.jpg", "image001.jpg"]
        inner = features.FeatureView(fset, Two)               # a second user keeps the data when the first leaves
        assert np.array_equal(view.get_feature_patch(1, 0).data, ref.fmap("image000.jpg").patches[0])
    assert fset.fmap("image000.jpg").is_loaded
    inner.close()
    assert not any(m.is_loaded for m in maps)

    full = features.FeatureView(fset, rec)
    prob_lazy, _ = ba.build_problem(rec, full, None, None, None, for_references=set(rec.points3D.keys()))
    prob_ref, _ = ba.build_problem(rec, features.FeatureView(ref, rec), None, None, None, for_references=set(rec.points3D.keys()))
    assert np.array_equal(np.asarray(prob_lazy.patches), np.asarray(prob_ref.patches))
    assert np.array_equal(prob_lazy.corner, prob_ref.corner) and np.array_equal(prob_lazy.obs_pt, prob_ref.obs_pt)
    del prob_lazy
    full.close()
    assert not any(m.is_loaded for m in maps)
    maps[0].lock()                                            # Lock(): resident for good
    features.FeatureView(fset, rec).close()
    assert maps[0].is_loaded and not any(m.is_loaded for m in maps[1:])


def test_lazy_cache_falls_back_to_eager_maps_where_metadata_needs_the_data(tmp_path):
    from pixsfm import features
    from pixsfm._pixsfm._features import LazyFeatureMap
    from pixsfm.features import store_features
    rng = np.random.default_rng(5)
    fm = features.FeatureManager([8], np.float16)
    fm.fset(0).emplace("a.jpg", features.FeatureMap(rng.normal(size=(3, 4, 4, 8)).astype(np.float16), [1, 2, 5], np.zeros((3, 2), np.int32),
                                                    {"scale": (1.0, 1.0), "is_sparse": True}))
    store_features.write_feature_manager_cache(tmp_path / "g.h5", fm, "grouped")
    got = store_features.load_features_from_cache(tmp_path / "g.h5", fill=False).fset(0).fmap("a.jpg")
    assert not isinstance(got, LazyFeatureMap) and np.array_equal(got.patches, fm.fset(0).fmap("a.jpg").patches)


def test_references_cache_round_trip(tmp_path):
    """features/store_references.py:14-58: one {point3D_id: Reference} map per level, observations and empty tracks included"""
    from pixsfm import features
    from pixsfm.features import store_references
    rng = np.random.default_rng(8)
    levels = []
    for lvl, ch in enumerate((16, 8)):
        refs = {}
        for pid in (3, 11, 400):
            r = features.Reference((pid % 7 + 1, pid % 5), rng.normal(size=(1, ch)))
            if pid != 11:
                r.observations = [rng.normal(size=(1, ch)) for _ in range(3)]
                r.costs = [0.1 * k for k in range(3)]
                r.track = [(1, 4), (2, 0), (5, 9)]
            refs[pid] = r
        levels.append(refs)
    store_references.write_references_cache(tmp_path / "refs.h5", levels)
    got = store_references.load_references_from_cache(tmp_path / "refs.h5")
    assert len(got) == 2 and all(sorted(g) == [3, 11, 400] for g in got)
    for a_map, b_map in zip(levels, got):
        for pid, a in a_map.items():
            b = b_map[pid]
            assert b.source == a.source and np.array_equal(a.descriptor, b.descriptor) and b.descriptor.dtype == np.float64
            assert len(b.observations) == len(a.observations) and all(np.array_equal(x, y) for x, y in zip(a.observations, b.observations))
            assert b.costs == [float(c) for c in a.costs] and b.track == (a.track or [])
