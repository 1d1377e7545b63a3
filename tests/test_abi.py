"""CPU-side checks of the boundary: the C-ABI library builds, loads, and exports every symbol the
header declares; host-only entry points agree with the oracle; the product never imports oracle/."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from hands_b200 import _lib
from oracle import geometry_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "hands_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = header_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/hands_b200.h but not exported"
    assert sorted(_lib.SYMBOLS) == names
    assert lib.hb_version() >= 100


def test_workspace_sizes_and_argument_errors():
    lib = _lib.load()
    assert lib.hb_mano_workspace_bytes(0, 0) == 0
    assert lib.hb_mano_workspace_bytes(1024, 1) > lib.hb_mano_workspace_bytes(1024, 0) > 0
    # per hand, in floats: forward A 192 + OFF 8 + feature slabs 2 x 152 + v_posed 2400 = 2904; the backward adds the
    # per-slice partials 5 x (192 + 8), the dL/dv_posed slabs 2 x 2400 and the split-K feature partials 4 x 160 = 6440
    assert lib.hb_mano_workspace_bytes(1024, 0) == 1024 * 11616
    assert lib.hb_mano_workspace_bytes(1024, 1) == 1024 * 37376
    assert lib.hb_pcl_bwd_workspace_bytes(8, 2, 3, 224) == 8 * 4 * 224 * 224 * 4  # one float4 gradient per intermediate pixel
    assert lib.hb_pcl_bwd_workspace_bytes(2 * 8192, 2, 3, 224) == 2 * 4096 * 4 * 224 * 224 * 4  # capped at 4096 images per chunk
    # argument validation happens before any CUDA call, so it is testable without a GPU
    rc = lib.hb_mano_head_fwd(None, None, 1, None, None, None, None, None, 4, 224.0, 0.1, None, None, None, None, None, None, None, 0, None)
    assert rc == -1 and b"NULL" in lib.hb_last_error_string()
    assert lib.hb_pcl_fwd(None, None, 3, 2, 3, 224, None, None) == -1
    assert lib.hb_matrix_to_axis_angle_fwd(None, 0, None, None) == 0
    # the rows either side of the path: same conventions (negative code + message, empty batches are no-ops)
    assert lib.hb_rot6d_to_rotmat_fwd(None, 4, 0, None, None) == -1 and lib.hb_rot6d_to_rotmat_fwd(None, 0, 7, None, None) == -1
    assert lib.hb_rot6d_to_rotmat_fwd(None, 0, 2, None, None) == 0
    rc = lib.hb_mano_head_fwd(None, None, 9, None, None, None, None, None, 4, 224.0, 0.1, None, None, None, None, None, None, None, 0, None)
    assert rc == -1
    assert lib.hb_kp_loss_fwd(None, None, None, None, None, None, None, None, 5, 224.0, None, None, None) == -1
    assert lib.hb_kp_loss_bwd(None, None, None, None, None, None, None, 0, None, None, None, None, None) == 0
    assert lib.hb_mrrpe(None, None, None, None, None, 3, None, None, None) == -1
    assert lib.hb_gt_process(None, None, None, None, 2, 224.0, None, None, None, None) == -1 and lib.hb_gt_process(None, None, None, None, 0, 224.0, None, None, None, None) == 0
    assert lib.hb_kpe_features(None, None, 3, 4, None, None, None, None, None) == -1 and lib.hb_kpe_features(None, None, 0, 4, None, None, None, None, None) == 0


def test_host_homography_matches_oracle(golden_dir):
    lib = _lib.load()
    g = np.load(os.path.join(golden_dir, "pcl.npz"))
    for j in range(8):
        bbox = np.ascontiguousarray(g["small_bbox"][j].astype(np.int32))
        K = np.ascontiguousarray(g["small_K"][j // 2].astype(np.float32))
        P = np.zeros(9, np.float32)
        R = np.zeros(9, np.float32)
        s = ctypes.c_int32()
        rc = lib.hb_pcl_homography_host(bbox.ctypes.data, K.ctypes.data, 64, P.ctypes.data, R.ctypes.data, ctypes.byref(s))
        assert rc == 0 and s.value == int(g["small_s"][j])
        assert np.array_equal(R.reshape(3, 3), g["small_rot"][j])
        Pref, _, _ = O.pcl_homography(bbox.tolist(), torch.from_numpy(K), 64)
        np.testing.assert_allclose(P.reshape(3, 3), Pref.numpy(), rtol=2e-7, atol=0)


def test_product_does_not_import_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "hands_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, os.path.join(dirpath, f)


def test_cpu_tensors_are_rejected_not_silently_computed():
    from hands_b200.common import rot, transforms

    with pytest.raises(RuntimeError, match="no CPU path"):
        rot.matrix_to_axis_angle(torch.eye(3)[None])
    with pytest.raises(RuntimeError, match="no CPU path"):
        transforms.project2d_batch(torch.eye(3)[None], torch.ones(1, 2, 3))
    with pytest.raises(RuntimeError, match="no CPU path"):
        rot.rot6d_to_rotmat(torch.ones(2, 6))
    with pytest.raises(RuntimeError, match="no CPU path"):
        rot.rotation_6d_to_matrix(torch.ones(2, 16, 6))
    from hands_b200.losses import keypoint_losses
    from hands_b200.pcl import kpe_features

    with pytest.raises(RuntimeError, match="no CPU path"):
        keypoint_losses(torch.zeros(2, 21, 3), torch.zeros(2, 21, 2), torch.zeros(2, 21, 3), torch.zeros(2, 21, 2), torch.ones(2, 21))
    with pytest.raises(RuntimeError, match="no CPU path"):
        kpe_features(torch.zeros(2, 4, dtype=torch.int32), torch.eye(3).repeat(2, 1, 1), 4)


def test_xdict_contract():
    from hands_b200.common.xdict import xdict

    d = xdict()
    d["a"] = 1
    with pytest.raises(AssertionError):
        d["a"] = 2
    assert list(d.postfix(".r").keys()) == ["a.r"] and list(d.prefix("mano.").keys()) == ["mano.a"]
    e = xdict({"b": 2})
    d.merge(e)
    assert sorted(d.keys()) == ["a", "b"]
    with pytest.raises(AssertionError):
        d.merge(e)


def test_stale_binary_detection_uses_source_digest(monkeypatch):
    """_lib.load() rebuilds when the sha256 of csrc/ + the header + the flags differs from the stamp written at build time
    (mtimes do not survive the copy to a GPU box; content does), and refuses a binary whose hb_version() is not the header's."""
    from hands_b200 import _build, _lib

    _build.build()
    assert not _build.needs_build()
    monkeypatch.setattr(_build, "NVCC_FLAGS", _build.NVCC_FLAGS + ["-DHB_SOMETHING_ELSE"])
    assert _build.needs_build()
    monkeypatch.undo()
    assert not _build.needs_build()
    assert _lib.load().hb_version() == _build.header_version() >= 201


def test_cpu_baseline_legs_run():
    """The CPU legs bench.py reports (scripts/bench_legs.py) stay runnable: per-sample loop, 1 thread, batched fixed-s."""
    import sys

    sys.path.insert(0, ROOT)
    from scripts import bench_legs as L

    v, dt = L.cpu_loop_all_threads(2, 1, 0)
    v1, _ = L.cpu_loop_one_thread(2)
    vb, _ = L.cpu_batched(2, 1, 0)
    assert v > 0 and v1 > 0 and vb > 0 and dt > 0
    c1 = L.config_c1()
    assert c1["hands_per_s"] > 0
