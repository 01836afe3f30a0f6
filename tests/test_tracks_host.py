"""Feature tracks without a GPU: the ``tracks`` config block, the C ABI of include/spn_tracks.h and the oracle
(oracle/tracks_oracle.py) on hand-built graphs with known answers."""
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import tracks_oracle as T


# ---------------------------------------------------------------------------------------------------------- config
def _config():
    import yaml
    return yaml.safe_load((ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "superpoint_match_tracks.yaml").read_text())


def test_tracks_config_defaults_and_absence():
    from superpoint_nerf_pytorch_b200.matching import tracks_config, verify_config
    cfg = _config()
    assert tracks_config(cfg) == {"min_length": 2}
    assert verify_config(cfg)["model"] == "fundamental"
    assert tracks_config({"verification": {"model": "homography"}, "tracks": {}}) == {"min_length": 2}
    assert tracks_config({"verification": {"model": "homography"}, "tracks": {"min_length": 5}}) == {"min_length": 5}
    assert tracks_config({}) is None and tracks_config({"tracks": None}) is None
    verify_cfg = ROOT / "superpoint-nerf-pytorch_b200" / "configs" / "superpoint_match_verify.yaml"
    import yaml
    assert tracks_config(yaml.safe_load(verify_cfg.read_text())) is None     # the verify config stays without tracks


def test_tracks_config_names_the_key():
    from superpoint_nerf_pytorch_b200.matching import tracks_config
    ver = {"model": "fundamental"}
    for key, value in (("min_len", 2), ("min_length", 1), ("min_length", 0), ("min_length", -3), ("min_length", True),
                       ("min_length", 2.5), ("min_length", 2.0), ("min_length", "2"), ("min_length", None)):
        with pytest.raises(ValueError, match=f"tracks.{key}"):
            tracks_config({"verification": ver, "tracks": {key: value}})
    with pytest.raises(ValueError, match="tracks: expected a mapping"):
        tracks_config({"verification": ver, "tracks": [2]})
    with pytest.raises(ValueError, match="tracks: needs a verification block"):
        tracks_config({"tracks": {"min_length": 2}})
    with pytest.raises(ValueError, match="tracks: needs a verification block"):
        tracks_config({"tracks": {}, "verification": None})


def test_cli_validates_the_tracks_block(tmp_path, monkeypatch):
    import yaml
    from superpoint_nerf_pytorch_b200 import matching as M
    monkeypatch.setenv("WORLD_SIZE", "1")
    for edit, key in ((lambda c: c["tracks"].update(min_length=1), "tracks.min_length"),
                      (lambda c: c.pop("verification"), "tracks: needs a verification block")):
        cfg = _config()
        edit(cfg)
        path = tmp_path / "bad.yaml"
        path.write_text(yaml.safe_dump(cfg))
        with pytest.raises(ValueError, match=key):
            M.main(config_path=str(path))


# ---------------------------------------------------------------------------------------------------------- oracle
def _table(edges, counts, min_length=2):
    off = np.r_[0, np.cumsum(counts)].astype(np.int64)
    lab = T.labels(np.asarray(edges, np.int64).reshape(-1, 2), int(off[-1]))
    return (lab, *T.tracks(lab, off, min_length))


def test_oracle_chain_and_star():
    # chain 0-1-2-3-4 over five images of one keypoint each, edges in descending order
    lab, off, obs, cons, tof = _table([(3, 4), (2, 3), (1, 2), (0, 1)], [1, 1, 1, 1, 1])
    assert lab.tolist() == [0] * 5 and off.tolist() == [0, 5] and cons.tolist() == [True]
    assert obs.tolist() == [[n, 0] for n in range(5)] and tof.tolist() == [0] * 5
    # star around row 5 (image 2, keypoint 1) over images of two keypoints: rows 1, 3, 5, 7
    lab, off, obs, cons, tof = _table([(5, 1), (7, 5), (5, 3)], [2, 2, 2, 2])
    assert lab.tolist() == [0, 1, 2, 1, 4, 1, 6, 1]
    assert off.tolist() == [0, 4] and obs.tolist() == [[0, 1], [1, 1], [2, 1], [3, 1]] and cons.tolist() == [True]
    assert tof.tolist() == [-1, 0, -1, 0, -1, 0, -1, 0]


def test_oracle_two_triangles_joined_by_one_edge():
    # triangle A = rows {0, 3, 6}, triangle B = rows {1, 4, 7}; three images of three keypoints
    tri = [(0, 3), (3, 6), (6, 0), (1, 4), (4, 7), (7, 1)]
    lab, off, obs, cons, tof = _table(tri, [3, 3, 3])
    assert off.tolist() == [0, 3, 6] and cons.tolist() == [True, True]
    assert obs.tolist() == [[0, 0], [1, 0], [2, 0], [0, 1], [1, 1], [2, 1]]
    assert tof.tolist() == [0, 1, -1, 0, 1, -1, 0, 1, -1]
    lab, off, obs, cons, tof = _table(tri + [(6, 4)], [3, 3, 3])      # one edge joins them: two per image
    assert lab.tolist() == [0, 0, 2, 0, 0, 5, 0, 0, 8] and off.tolist() == [0, 6] and cons.tolist() == [False]
    assert obs.tolist() == [[0, 0], [0, 1], [1, 0], [1, 1], [2, 0], [2, 1]]
    # min_length drops the small components and renumbers the rest
    lab, off, obs, cons, tof = _table(tri + [(2, 5)], [3, 3, 3], min_length=3)
    assert off.tolist() == [0, 3, 6] and tof.tolist() == [0, 1, -1, 0, 1, -1, 0, 1, -1]


def test_oracle_conflict_within_one_image_duplicates_and_self_loops():
    # rows 0, 1 in image 0 (two keypoints), row 2 in image 1: 0-2-1 puts two keypoints of image 0 into one track
    lab, off, obs, cons, tof = _table([(0, 2), (2, 1), (2, 1), (1, 2), (0, 0), (2, 2)], [2, 1, 1])
    assert lab.tolist() == [0, 0, 0, 3] and off.tolist() == [0, 3] and cons.tolist() == [False]
    assert obs.tolist() == [[0, 0], [0, 1], [1, 0]] and tof.tolist() == [0, 0, 0, -1]
    # duplicates and self-loops alone change nothing
    lab2, *rest = _table([(0, 2), (0, 2), (2, 0), (1, 1), (3, 3)], [2, 1, 1])
    assert lab2.tolist() == [0, 1, 0, 3] and rest[0].tolist() == [0, 2] and rest[2].tolist() == [True]
    # no edges: all singletons, no tracks; an image without keypoints between two others
    lab, off, obs, cons, tof = _table(np.zeros((0, 2)), [2, 0, 3])
    assert lab.tolist() == [0, 1, 2, 3, 4] and off.tolist() == [0] and obs.shape == (0, 2) and (tof == -1).all()
    lab, off, obs, cons, tof = _table([(1, 4)], [2, 0, 3])
    assert obs.tolist() == [[0, 1], [2, 2]] and cons.tolist() == [True]


def test_oracle_match_edges_and_keep():
    counts, pairs = [2, 3, 1], [(0, 1), (1, 2), (0, 2)]
    offsets = [0, 2, 3, 4]
    matches = [(0, 2), (1, 0), (2, 0), (1, 0)]
    edges, off = T.match_edges(counts, pairs, offsets, matches)
    assert off.tolist() == [0, 2, 5, 6] and edges.tolist() == [[0, 4], [1, 2], [4, 5], [1, 5]]
    t_off, obs, cons, tof, lab = T.build_tracks(counts, pairs, offsets, matches, keep=[True, True, True, False])
    assert lab.tolist() == [0, 1, 1, 3, 0, 0] and t_off.tolist() == [0, 3, 5] and cons.tolist() == [True, True]
    assert obs.tolist() == [[0, 0], [1, 2], [2, 0], [0, 1], [1, 0]] and tof.tolist() == [0, 1, 1, -1, 0, 0]
    t_off, obs, cons, tof, lab = T.build_tracks(counts, pairs, offsets, matches)      # all: keypoints 0 and 1 of image 0
    assert lab.tolist() == [0, 0, 0, 3, 0, 0] and t_off.tolist() == [0, 5] and cons.tolist() == [False]
    assert not T.build_tracks(counts, pairs, offsets, matches, keep=[False] * 4)[0][1:].size


# ---------------------------------------------------------------------------------------------------------- C ABI
@pytest.fixture(scope="module")
def built_lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("spn_build", ROOT / "superpoint-nerf-pytorch_b200" / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def test_cabi_exports_the_tracks_symbols(built_lib):
    import ctypes
    from superpoint_nerf_pytorch_b200 import _native as N
    text = (ROOT / "include" / "spn_tracks.h").read_text()
    assert sorted(re.findall(r"SPN_API\s+\w+\s+(\w+)\s*\(", text)) == sorted(N.TRACKS_PROTOTYPES) == \
        ["spn_track_labels", "spn_track_table"]
    others = (set(N.PROTOTYPES) | set(N.JPEG_PROTOTYPES) | set(N.NERF_PROTOTYPES) | set(N.POSED_PROTOTYPES)
              | set(N.MATCH_PROTOTYPES) | set(N.RETRIEVAL_PROTOTYPES) | set(N.VERIFY_PROTOTYPES))
    assert not set(N.TRACKS_PROTOTYPES) & others
    lib = ctypes.CDLL(str(built_lib))
    assert all(hasattr(lib, name) for name in N.TRACKS_PROTOTYPES)


def test_tracks_reject_null_and_out_of_range_arguments(built_lib):
    """A NULL context and out-of-range values -> SPN_E_INVALID (-1) and a message, before any CUDA call (child process;
    the stand-in context and buffers are never dereferenced on these paths)."""
    code = r'''
import sys, ctypes as C
sys.path.insert(0, %r)
from superpoint_nerf_pytorch_b200 import _native as N
lib = N.load_library()
fake = C.create_string_buffer(64)
def labels(ctx=fake, edges=fake, E=4, K=8, resume=0, label=fake, bad=fake):
    return lib.spn_track_labels(ctx, edges, E, K, resume, label, bad, None), lib.spn_last_error().decode()
def table(ctx=fake, label=fake, K=8, off=fake, N_=2, ml=2, toff=fake, obs=fake, cons=fake, tof=fake, tot=fake, bad=fake):
    rc = lib.spn_track_table(ctx, label, K, off, N_, ml, toff, obs, cons, tof, tot, bad, None)
    return rc, lib.spn_last_error().decode()
cases = [(labels, dict(ctx=None), "null pointer (ctx)"), (labels, dict(K=0), "K = 0"), (labels, dict(K=-5), "K = -5"),
         (labels, dict(E=-1), "E = -1"), (labels, dict(resume=2), "resume = 2"), (labels, dict(label=None), "null pointer"),
         (labels, dict(bad=None), "null pointer"), (labels, dict(edges=None), "null pointer (edges with E = 4)"),
         (table, dict(ctx=None), "null pointer (ctx)"), (table, dict(K=0), "K = 0"), (table, dict(K=-1), "K = -1"),
         (table, dict(N_=0), "N = 0"), (table, dict(N_=-2), "N = -2"), (table, dict(ml=1), "min_length = 1"),
         (table, dict(ml=0), "min_length = 0"), (table, dict(ml=-7), "min_length = -7")]
for key in ("label", "off", "toff", "obs", "tof", "tot", "bad", "cons"):
    cases.append((table, {key: None}, "null pointer"))
for fn, kw, msg in cases:
    rc, err = fn(**kw)
    assert rc == -1 and msg in err, (fn.__name__, kw, rc, err)
# E == 0 with NULL edges passes the edges check: the next check (label / bad) is the one that fails
rc, err = labels(E=0, edges=None, label=None)
assert rc == -1 and "null pointer (label / bad)" in err, (rc, err)
print("checked", len(cases) + 1)
''' % str(ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "checked 25" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
