"""CPU tests (no GPU): the C ABI loads and exports what include/agt.h declares, host-side logic,
and the multi-GPU partition / gather logic over gloo with world_size 2."""
import os
import re
import socket
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from accurate_aprilgroup_tracking_b200 import _lib, sharding, synth

ROOT = Path(__file__).resolve().parent.parent


# ---------------------------------------------------------------------------- C ABI
def test_library_exports_every_declared_symbol(lib_built):
    header = (ROOT / "include" / "agt.h").read_text()
    declared = set(re.findall(r"\b(agt_[a-z0-9_]+)\s*\(", header))
    declared -= {"agt_status"}
    assert len(declared) >= 25
    nm = subprocess.run(["nm", "-D", "--defined-only", str(lib_built)], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (agt_[a-z0-9_]+)", nm))
    assert declared <= exported, f"declared but not exported: {sorted(declared - exported)}"
    assert declared == set(_lib.PROTOTYPES), f"ctypes prototypes out of sync: {sorted(declared ^ set(_lib.PROTOTYPES))}"
    lib = _lib.load()
    assert lib.agt_version() == 100


def test_library_is_sm100a_only(lib_built):
    from accurate_aprilgroup_tracking_b200 import _build
    cuobjdump = Path(_build._nvcc()).with_name("cuobjdump")       # the toolkit that built the library, on PATH or not
    out = subprocess.run([str(cuobjdump), "--list-elf", str(lib_built)], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = set(re.findall(r"sm_\d+a?", out.stdout))
    assert archs == {"sm_100a"}, archs


def test_no_cpu_fallback_without_device(lib_built):
    """Without a CUDA device the product path must fail loudly (never route through the oracle)."""
    import ctypes as C
    lib = _lib.load()
    if lib.agt_device_count() > 0:
        pytest.skip("a GPU is visible")
    h = C.c_void_p()
    rc = lib.agt_create(0, C.byref(h))
    assert rc == _lib.AGT_ERR_NO_DEVICE
    assert b"no CPU fallback" in lib.agt_last_error(None)
    from accurate_aprilgroup_tracking_b200 import cv_compat
    with pytest.raises(RuntimeError):
        cv_compat.HostContext(0)
    with pytest.raises(RuntimeError):
        cv_compat.solvePnP(np.zeros((8, 3), np.float32), np.zeros((8, 2), np.float32), np.eye(3), None)


def test_product_does_not_import_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    pkg = ROOT / "accurate_aprilgroup_tracking_b200"
    for f in pkg.rglob("*.py"):
        txt = f.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M), f
        assert "cv2.solvePnP" not in txt and "calcOpticalFlowPyrLK(" not in txt.replace("self._agt.calcOpticalFlowPyrLK(", "") \
            .replace("def calcOpticalFlowPyrLK(", "").replace("default_context().calcOpticalFlowPyrLK(", ""), f


def test_null_context_is_rejected(lib_built):
    lib = _lib.load()
    assert lib.agt_sync(None) == _lib.AGT_ERR_INVALID
    assert lib.agt_destroy(None) == _lib.AGT_ERR_INVALID
    assert lib.agt_launch_count(None) == -1


# ---------------------------------------------------------------------------- host logic
def test_rodrigues_matches_opencv():
    import cv2
    from accurate_aprilgroup_tracking_b200 import cv_compat
    rng = np.random.default_rng(0)
    for _ in range(50):
        r = rng.normal(0, 1.0, 3)
        for dt in (np.float64, np.float32):
            ours = cv_compat.Rodrigues(r.astype(dt).reshape(3, 1))[0]
            ref = cv2.Rodrigues(r.astype(dt).reshape(3, 1))[0]
            assert ours.dtype == ref.dtype and ours.shape == (3, 3)
            assert np.abs(ours - ref).max() < (1e-6 if dt == np.float32 else 1e-12)
        back = cv_compat.Rodrigues(cv2.Rodrigues(r)[0])[0]
        assert back.shape == (3, 1) and np.abs(back.ravel() - cv2.Rodrigues(cv2.Rodrigues(r)[0])[0].ravel()).max() < 1e-9
    near_pi = np.array([3.1, 0.02, -0.01])
    assert np.abs(cv_compat.Rodrigues(cv2.Rodrigues(near_pi)[0])[0].ravel() - near_pi).max() < 1e-6


def test_bgr_to_gray_bit_exact():
    import cv2
    from accurate_aprilgroup_tracking_b200.aprilgroup_pose_estimation.detect_pose import bgr_to_gray
    rng = np.random.default_rng(1)
    img = rng.integers(0, 256, (120, 160, 3), dtype=np.uint8)
    assert np.array_equal(bgr_to_gray(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))


def test_transform_helper_matches_reference_formulas():
    from accurate_aprilgroup_tracking_b200.aprilgroup_pose_estimation.transform_helper import TransformHelper as TH
    from oracle import ape_oracle
    rng = np.random.default_rng(2)
    for _ in range(20):
        m = synth.rodrigues(rng.normal(0, 0.8, 3))
        e = TH.rotation_matrix_to_euler_angles(m)
        assert np.allclose(e, ape_oracle.euler_from_rotation(m))
        assert np.allclose(TH.euler_angles_to_rotation_matrix(e), m, atol=1e-12)
    pts = TH.get_initial_pts(0.02)
    assert pts.tolist() == [[-0.01, -0.01, 0.0], [-0.01, 0.01, 0.0], [0.01, 0.01, 0.0], [0.01, -0.01, 0.0]]
    size, tvec, rvec = ape_oracle.group_from_json(synth.april_group_dict())[5]
    ours = TH.transform_marker_corners(pts, (rvec, tvec))
    assert np.abs(ours - ape_oracle.tag_object_points(size, rvec, tvec)).max() < 1e-8
    assert TH.get_rmat_tvec(np.eye(4))[1].dtype == np.float32
    with pytest.raises(ValueError):
        TH.transform_marker_corners(pts, (np.zeros(0), tvec))


def test_synthetic_world_geometry():
    n = synth.face_normals()
    assert n.shape == (12, 3) and np.allclose(np.linalg.norm(n, axis=1), 1.0)
    assert len({tuple(np.round(v, 6)) for v in n}) == 12
    obj = synth.object_points()
    assert obj.shape == (48, 3)
    for k in range(12):                       # corners lie on their face plane, 20 mm apart
        c = obj[4 * k:4 * k + 4]
        assert np.allclose(c @ n[k], synth.INRADIUS, atol=1e-6)
        assert np.allclose(np.linalg.norm(c[1] - c[0]), synth.TAG_SIZE, atol=1e-6)
    s, tg, nn, cc = synth.surface_model()
    assert s.shape == (12 * 41 * 41, 4) and tg.max() == 11 and np.all(np.diff(tg.astype(int)) >= 0)
    tr = synth.trajectory(1, 300)
    d = np.abs(np.diff(tr, axis=0))
    assert d[:, :3].max() < 0.03 and d[:, 3:].max() < 0.003 and not (d == 0).any()


def test_cv_compat_level_rule_matches_opencv():
    import cv2
    from accurate_aprilgroup_tracking_b200.cv_compat import HostContext
    for (w, h) in [(640, 480), (1920, 1080), (320, 240), (100, 80), (60, 50), (30, 30)]:
        img = np.zeros((h, w), np.uint8)
        max_level, _ = cv2.buildOpticalFlowPyramid(img, (21, 21), 3, withDerivatives=False)
        assert HostContext._levels_for(w, h, 3) == max_level + 1, (w, h)


# ---------------------------------------------------------------------------- multi-GPU partition logic (gloo)
def test_frame_block_partition():
    for n in (0, 1, 7, 4096, 4099):
        for world in (1, 2, 3, 8):
            blocks = [sharding.frame_block(n, r, world) for r in range(world)]
            assert blocks[0][0] == 0 and blocks[-1][1] == n
            assert all(blocks[i][1] == blocks[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in blocks]
            assert max(sizes) - min(sizes) <= 1
    assert sharding.local_streams(64, 3, 8) == list(range(3, 64, 8))
    with pytest.raises(ValueError):
        sharding.frame_block(10, 2, 2)


_WORKER = r"""
import sys, os
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
from accurate_aprilgroup_tracking_b200 import sharding
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
n = 11
full = torch.arange(n * 6, dtype=torch.float64).reshape(n, 6)
a, b = sharding.frame_block(n, rank, world)
got = sharding.gather_poses(full[a:b].clone(), n)
assert torch.equal(got, full), (rank, got)
ids = sharding.local_streams(7, rank, world)
got2 = sharding.gather_stream_poses(full[:7][ids].clone(), 7)
assert torch.equal(got2, full[:7]), (rank, got2)
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_gather_poses_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=str(ROOT)))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script)]
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("ok") == 2


def test_numa_binding_helpers(tmp_path, monkeypatch):
    """sharding.on_gpu_numa_node: sysfs cpulist parsing, the CPU set is restored afterwards, unknown topology is a no-op."""
    import os
    import types
    from accurate_aprilgroup_tracking_b200 import sharding
    assert sharding.parse_cpulist("0-3,8,10-11\n") == [0, 1, 2, 3, 8, 10, 11]
    assert sharding.parse_cpulist("") == []
    before = os.sched_getaffinity(0)
    # no GPU here: the topology is unknown and nothing changes
    with sharding.on_gpu_numa_node(0, sysfs=str(tmp_path)) as node:
        assert node is None and os.sched_getaffinity(0) == before
    # a fake sysfs tree + device properties: the thread runs on the node's CPUs inside the block only
    import torch
    props = types.SimpleNamespace(pci_domain_id=0, pci_bus_id=0x1b, pci_device_id=0)
    monkeypatch.setattr(torch.cuda, "get_device_properties", lambda i: props)
    dev = tmp_path / "bus/pci/devices/0000:1b:00.0"
    dev.mkdir(parents=True)
    (dev / "numa_node").write_text("1\n")
    nd = tmp_path / "devices/system/node/node1"
    nd.mkdir(parents=True)
    one = min(before)
    (nd / "cpulist").write_text(f"{one}\n")
    with sharding.on_gpu_numa_node(0, sysfs=str(tmp_path)) as node:
        assert node == 1 and os.sched_getaffinity(0) == {one}
    assert os.sched_getaffinity(0) == before
    (dev / "numa_node").write_text("-1\n")
    with sharding.on_gpu_numa_node(0, sysfs=str(tmp_path)) as node:
        assert node is None


def test_pack_detections_maps_tag_ids_to_their_position_in_the_group():
    """A real april_group.json has arbitrary ids in arbitrary key order: corner index = 4 * (position of the tag in the JSON)
    + j (detect_pose.py:122, :202), and the reference looks object points up by id (detect_pose.py:405-437).  The packed
    layout must therefore go by position, not by id (round 1 wrote to slot 4 * id)."""
    from accurate_aprilgroup_tracking_b200.batched import pack_detections, tag_positions
    ids = [7, 3, 42, 19]                                   # JSON key order
    c = lambda v: np.full((4, 2), float(v)) + np.arange(8).reshape(4, 2)
    dets = [[(42, c(420)), (7, c(70))], [(19, c(190))], []]
    img, valid, n = pack_detections(dets, ids)
    assert img.shape == (3, 16, 2) and valid.shape == (3, 16) and n.tolist() == [2, 1, 0]
    assert np.array_equal(img[0, 8:12], c(420)) and np.array_equal(img[0, 0:4], c(70))       # 42 is the third tag, 7 the first
    assert valid[0].tolist() == [1] * 4 + [0] * 4 + [1] * 4 + [0] * 4
    assert np.array_equal(img[1, 12:16], c(190)) and valid[1].tolist() == [0] * 12 + [1] * 4
    with pytest.raises(KeyError):                          # unknown id: the reference's extrinsics[tag_id] raises KeyError too
        pack_detections([[(5, c(0))]], ids)
    with pytest.raises(ValueError):
        tag_positions([1, 2, 1])
    # default = the synthetic dodecahedron, ids 0..11 in order
    img, valid, n = pack_detections([[(11, c(1))]])
    assert img.shape == (1, 48, 2) and valid[0, 44:].all() and n[0] == 1
    # the same tag reported twice fills one slot
    assert pack_detections([[(3, c(1)), (3, c(2))]], ids)[2][0] == 1
