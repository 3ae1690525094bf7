"""CPU: the product's host-side loader (Forest::load / Tree::load restatement + packed image) against the oracle's
independent parser, on synthetic archives always and on the 115 shipped archives when CRF_REFERENCE names a checkout of
the reference project."""
import ctypes as C
import shutil
from pathlib import Path

import numpy as np
import pytest

from conftest import REF_DATA


def _same_trees(gm, om, which, trees):
    for t in trees:
        a, b = gm.tree_dump(which, t), om.tree_dump(which, t)
        assert a.shape == b.shape
        leaf = b[:, 0] == 1
        assert np.array_equal(a[:, [0, 1, 15]], b[:, [0, 1, 15]])
        assert np.array_equal(a[~leaf][:, 2:14], b[~leaf][:, 2:14])
        assert np.array_equal(a[leaf][:, 14], b[leaf][:, 14])


def test_synthetic_archives_parse_identically(synth_models):
    gm, om = synth_models
    assert gm.info["hp_nodes"] == om.info["hp_nodes"] and gm.info["mp_nodes"] == om.info["mp_nodes"]
    assert gm.info["hp_leaves"] == om.info["hp_leaves"] and gm.info["mp_leaves"] == om.info["mp_leaves"]
    _same_trees(gm, om, -1, range(15))
    for f in range(5):
        _same_trees(gm, om, f, range(0, 20, 3))


def test_packed_roundtrip(crf, O, synth_models, tmp_path):
    gm, om = synth_models
    p = tmp_path / "m.crfb200"
    gm.save_packed(str(p))
    g2 = crf.Model(packed=str(p))
    o2 = O.Model(packed=str(p))
    assert g2.info == gm.info
    for which, n in [(-1, 15), (2, 20)]:
        for t in range(0, n, 4):
            assert np.array_equal(g2.tree_dump(which, t), gm.tree_dump(which, t))
            assert np.array_equal(o2.tree_dump(which, t), om.tree_dump(which, t))
            assert np.array_equal(o2.leaf_dump(which, t), om.leaf_dump(which, t))
    raw = bytearray(p.read_bytes())
    raw[len(raw) // 2] ^= 0x40
    (tmp_path / "bad.crfb200").write_bytes(bytes(raw))
    with pytest.raises(crf.CrfError) as e:
        crf.Model(packed=str(tmp_path / "bad.crfb200"))
    assert e.value.code == -3 and "checksum" in str(e.value)


def test_loader_errors_mirror_forest_load(crf, synth_dirs, tmp_path):
    hp, ffd = synth_dirs
    # missing directory / missing tree file -> CRF_ERR_IO ("File not found", include/Tree.hpp:202)
    with pytest.raises(crf.CrfError) as e:
        crf.Model(str(tmp_path / "nope"), ffd)
    assert e.value.code == -2
    part = tmp_path / "hp_part"
    shutil.copytree(hp, part)
    (part / "tree_007.txt").unlink()
    with pytest.raises(crf.CrfError) as e:
        crf.Model(str(part), ffd)
    assert e.value.code == -2 and "tree_007" in str(e.value)
    # fewer trees requested than present is fine (Forest::load reads tree_000..tree_{ntrees-1}, include/Forest.hpp:116-127)
    m = crf.Model(str(part), ffd, 7, 20)
    assert m.info["hp_trees"] == 7
    # truncated archive -> CRF_ERR_FORMAT
    trunc = tmp_path / "hp_trunc"
    shutil.copytree(hp, trunc)
    txt = (trunc / "tree_003.txt").read_text()
    (trunc / "tree_003.txt").write_text(txt[: len(txt) // 2])
    with pytest.raises(crf.CrfError) as e:
        crf.Model(str(trunc), ffd)
    assert e.value.code == -3
    # unfinished tree (i_node != m_num_nodes) is rejected (include/Tree.hpp:72-79, include/Forest.hpp:142-152)
    from face_alignment_cvpr_2012_b200 import synthetic_model as sm
    unf = tmp_path / "hp_unf"
    shutil.copytree(hp, unf)
    (unf / "tree_001.txt").write_text(sm.tree_text("hp", 6, np.random.default_rng(1), finished=False))
    with pytest.raises(crf.CrfError) as e:
        crf.Model(str(unf), ffd)
    assert e.value.code == -3 and "not finished" in str(e.value)
    # not an archive at all
    junk = tmp_path / "hp_junk"
    shutil.copytree(hp, junk)
    (junk / "tree_000.txt").write_text("hello world")
    with pytest.raises(crf.CrfError):
        crf.Model(str(junk), ffd)
    # wrong face size is outside the device layout
    odd = tmp_path / "hp_odd"
    shutil.copytree(hp, odd)
    for i in range(15):
        (odd / f"tree_{i:03d}.txt").write_text(sm.tree_text("hp", 5, np.random.default_rng(i), face_size=100))
    with pytest.raises(crf.CrfError) as e:
        crf.Model(str(odd), ffd)
    assert e.value.code == -6


def test_jungle_is_sorted_subdirectories(crf, synth_dirs, tmp_path):
    """FaceForest::FaceForest enumerates sub-directories and sorts them (src/FaceForest.cpp:39-44)."""
    hp, ffd = synth_dirs
    j = tmp_path / "jungle"
    for name, src in [("e_last", "forest_4"), ("a_first", "forest_0"), ("c", "forest_2"), ("b", "forest_1"), ("d", "forest_3")]:
        shutil.copytree(Path(ffd) / src, j / name)
    (j / "stray_file.txt").write_text("ignored")
    a, b = crf.Model(hp, str(j)), crf.Model(hp, ffd)
    for f in range(5):
        assert np.array_equal(a.tree_dump(f, 0), b.tree_dump(f, 0))


@pytest.mark.skipif(REF_DATA is None or not (REF_DATA / "trees_ffd").exists(), reason="no reference checkout (CRF_REFERENCE)")
def test_shipped_archives(crf, O):
    gm = crf.Model(str(REF_DATA / "trees_headpose"), str(REF_DATA / "trees_ffd"), 15, 20)
    om = O.Model(str(REF_DATA / "trees_headpose"), str(REF_DATA / "trees_ffd"), 15, 20)
    assert gm.info["hp_nodes"] == 176841 and gm.info["mp_nodes"] == 1536652  # SURVEY Appendix C
    assert gm.info["hp_leaves"] == 88428 and gm.info["mp_leaves"] == 768376
    _same_trees(gm, om, -1, range(15))
    for f in range(5):
        _same_trees(gm, om, f, range(20))
    # the staged packed image (what travels to the GPU box) holds exactly the oracle's text parse, leaves included
    from face_alignment_cvpr_2012_b200 import workloads as wl
    p = wl.staged_model_path()
    if p is not None:
        op = O.Model(packed=str(p))
        for which, n in [(-1, 15), (0, 20), (1, 20), (2, 20), (3, 20), (4, 20)]:
            for t in range(n):
                assert np.array_equal(op.tree_dump(which, t), om.tree_dump(which, t))
                assert np.array_equal(op.leaf_dump(which, t), om.leaf_dump(which, t))


def test_config_file_parser(crf):
    """data/config_ffd.txt of a reference checkout when one is named, else tests/golden/config_ffd.txt: the same entries in the
    same label / value layout (src/face_utils.cpp:50-140)."""
    cfg = REF_DATA / "config_ffd.txt" if REF_DATA is not None else None
    if cfg is None or not cfg.exists():
        cfg = Path(__file__).resolve().parent / "golden" / "config_ffd.txt"
    p = crf.loadConfigFile(str(cfg))
    assert (p.ntrees, p.max_depth, p.face_size, p.features, p.tree_path) == (20, 20, 125, [0, 1, 2], "data/trees_ffd")
    assert p.getPatchSize() == 31 and p.image_path.endswith("lfw_ffd_ann.txt")


def test_device_record_forms_agree(crf, synth_models, tmp_path):
    """pack.cc without a GPU: the wide, compact and shared-memory-window node records describe the same tests (crf_model_check_packing),
    for the synthetic forests, for forests with 30x30 rectangles, and for the shipped forests when they are staged."""
    import ctypes as C
    from face_alignment_cvpr_2012_b200 import capi, synthetic_model as sm, workloads as wl
    def check(model):
        hp, ffd = C.c_int(-1), C.c_int(-1)
        n = capi.lib().crf_model_check_packing(model.h, C.byref(hp), C.byref(ffd))
        assert n > 0, capi.lib().crf_last_error()
        return n, hp.value, ffd.value
    n, hp, ffd = check(synth_models[0])
    assert n == synth_models[0].info["hp_nodes"] + synth_models[0].info["mp_nodes"] and 0 < hp <= 30 and 0 < ffd <= 30
    big = crf.Model(*sm.write_model(tmp_path / "big", seed=3, hp_depth=6, ffd_depth=6, max_rect=30), 15, 20)
    assert check(big)[1] <= 30
    p = wl.staged_model_path()
    if p is not None:
        n, hp, ffd = check(crf.Model(packed=str(p)))
        assert (hp, ffd) == (30, 30) and n == 176841 + 1536652   # SURVEY Appendix C node counts; extents as measured in DESIGN 4.1


def test_feature_lists_and_channel_validation(crf, O, tmp_path):
    """ForestParam::features drives the plane layout (src/ImageSample.cpp:77-90): a model is accepted only if every split reads
    a plane its feature list provides — the reference would index m_feature_channels out of bounds, the GPU would read the
    next face's planes."""
    from face_alignment_cvpr_2012_b200 import synthetic_model as sm
    # all six feature kinds: 1 + 35 + 2 + 2 + 1 + 1 = 42 planes, splits read channels 0..41
    hp, ffd = sm.write_model(tmp_path / "all", seed=3, hp_trees=4, hp_depth=6, ffd_trees=3, ffd_depth=6, channels=42, features=(5, 0, 3, 1, 4, 2))
    m = crf.Model(hp, ffd, 4, 3)
    assert m.features == [0, 1, 2, 3, 4, 5] and m.info["num_channels"] == 42
    # the same trees under the shipped configuration (features 0 1 2 -> 38 planes) read planes that do not exist
    with pytest.raises(crf.CrfError) as e:
        m.set_features([0, 1, 2])
    assert e.value.code == -6 and "feature channel" in str(e.value)
    assert m.features == [0, 1, 2, 3, 4, 5]   # a rejected list leaves the model unchanged
    # archives that store features {0, 2} (3 planes) but whose splits read channel 30: rejected at load, text and packed alike
    hp2, ffd2 = sm.write_model(tmp_path / "bad", seed=4, hp_trees=2, hp_depth=5, ffd_trees=2, ffd_depth=5, channels=38, features=(0, 2))
    with pytest.raises(crf.CrfError) as e:
        crf.Model(hp2, ffd2, 2, 2)
    assert e.value.code == -6
    # ... and accepted when the splits stay inside the 3 planes; the run-time list may add planes but not remove used ones
    hp3, ffd3 = sm.write_model(tmp_path / "ok", seed=5, hp_trees=2, hp_depth=5, ffd_trees=2, ffd_depth=5, channels=3, features=(0, 2))
    m3 = crf.Model(hp3, ffd3, 2, 2)
    assert m3.features == [0, 2] and m3.info["num_channels"] == 3
    m3.set_features([2, 0, 3])
    assert m3.features == [0, 2, 3] and m3.info["num_channels"] == 5
    for bad in ([0, 0], [7], []):
        with pytest.raises(crf.CrfError):
            m3.set_features(bad)
    p = tmp_path / "m3.crfb200"
    crf.Model(hp3, ffd3, 2, 2).save_packed(str(p))
    assert crf.Model(packed=str(p)).features == [0, 2]


def test_single_forest_models_and_leaf_dump(crf, O, synth_dirs, synth_models):
    """Forest<S>::load on its own (include/Forest.hpp:103-129) and the leaf payloads (HeadPoseLeaf / MPLeaf)."""
    hp, ffd = synth_dirs
    gm, om = synth_models
    one = crf.Model(forest_dir=hp, kind="hp", ntrees=15)
    assert one.info["hp_trees"] == 15 and one.info["mp_forests"] == 0
    two = crf.Model(forest_dir=str(Path(ffd) / "forest_3"), kind="mp", ntrees=20)
    assert two.info["hp_trees"] == 0 and two.info["mp_forests"] == 1 and two.info["mp_trees"] == 20
    assert np.array_equal(two.tree_dump(0, 7), gm.tree_dump(3, 7))
    for which, t in [(-1, 0), (-1, 14), (0, 0), (4, 19)]:
        a, b = gm.leaf_dump(which, t), om.leaf_dump(which, t)
        assert a.shape == b.shape and np.array_equal(a, b)
    assert np.array_equal(two.leaf_dump(0, 5), gm.leaf_dump(3, 5))
    with pytest.raises(crf.CrfError):
        crf.Model(forest_dir=str(Path(hp) / "missing"), kind="hp", ntrees=15)
