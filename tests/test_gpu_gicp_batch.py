"""Batched GICP registration against one target (b200reg_gicp_align_batch / _device). Every registration of a batch must be
BITWISE the registration b200reg_align performs for the same (source, guess): the batch keeps the single path's covariance
kernel body, its correspondence kernels, the single inner launch's partition of the correspondences into chunks, every
summation order, and the host-side outer-loop arithmetic. The last test (the C layout of the result record) needs no GPU."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def b200():
    import torch

    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the gpu tests must run on the B200 box (there is no CPU fallback)")
    import lidarslam_ros2_b200 as m

    return m


def _engine(m, tgt, corr_dist=5.0):
    g = m.GeneralizedIterativeClosestPoint()
    g.setMaxCorrespondenceDistance(corr_dist)
    g.setInputTarget(tgt)
    return g


def _scans_and_guesses(src, n, seed=7):
    """n different (scan, guess) problems from one scan: sub-sampled / perturbed copies (ragged sizes) and perturbed guesses."""
    from lidarslam_ros2_b200 import synth

    rng = np.random.default_rng(seed)
    scans, guesses = [], []
    d = np.pi / 180
    for k in range(n):
        keep = rng.random(len(src)) < (1.0 - 0.07 * (k % 4))
        s = src[keep].copy()
        s[:, :3] += rng.normal(0, 0.004, size=(len(s), 3)).astype(np.float32)
        scans.append(np.ascontiguousarray(s[:, :3]))
        guesses.append(synth.pose_matrix((0.05 * (k % 3), -0.04 * (k % 2), 0.0), (0, 0, 0.3 * d * (k % 5))).astype(np.float32))
    return scans, guesses


def _single(g, scans, guesses):
    """setInputSource + align(guess) one after the other: (pose, converged, iterations, evaluations, correspondences)."""
    out = []
    for s, T in zip(scans, guesses):
        g.setInputSource(s)
        P = g.align(T)
        st = g.stats()
        out.append((P, g.hasConverged(), st["iterations"], st["evaluations"], g.numCorrespondences()))
    return out


def _assert_equal(r, ref, tag=""):
    assert len(r["pose"]) == len(ref)
    for k, (P, conv, it, ev, m) in enumerate(ref):
        assert r["status"][k] == 0, (tag, k, r["status"][k])
        assert np.array_equal(r["pose"][k], P, equal_nan=True), (tag, k, np.abs(r["pose"][k] - P).max())
        assert bool(r["converged"][k]) == conv and r["iterations"][k] == it, (tag, k)
        assert r["evaluations"][k] == ev and r["correspondences"][k] == m, (tag, k, r["evaluations"][k], ev)


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["tiny", "small", "c1"])
def test_gicp_batch_equals_single_bitwise(b200, config):
    from lidarslam_ros2_b200 import synth

    src, tgt, _ = synth.registration_pair(config, 2.0)
    g = _engine(b200, tgt)
    scans, guesses = _scans_and_guesses(src, 9 if config != "c1" else 7)
    ref = _single(g, scans, guesses)
    for slots in (3, 2, 1):
        g.setBatchSlots(slots)
        r = g.alignBatch(scans, guesses)
        _assert_equal(r, ref, (config, slots))
        # the handle's getters describe the last registration; the stats sum over the batch
        assert np.array_equal(g.getFinalTransformation(), ref[-1][0])
        assert g.hasConverged() == ref[-1][1] and g.numCorrespondences() == ref[-1][4]
        st = g.stats()
        assert st["iterations"] == ref[-1][2]
        assert st["evaluations"] == sum(x[3] for x in ref)
        assert st["gicp_inner_launches"] >= max(x[2] for x in ref) and st["gicp_pair_evaluations"] > 0


@pytest.mark.gpu
def test_gicp_batch_device_sources_identity_guess(b200):
    import torch

    from lidarslam_ros2_b200 import synth

    src, tgt, _ = synth.registration_pair("small", 2.0)
    g = _engine(b200, tgt)
    scans, _ = _scans_and_guesses(src, 5, seed=11)
    ref = _single(g, scans, [None] * len(scans))
    dev = [torch.from_numpy(np.concatenate([s, np.ones((len(s), 1), np.float32)], axis=1)).cuda() for s in scans]
    torch.cuda.synchronize()
    r = g.alignBatchDevice([d.data_ptr() for d in dev], [d.shape[0] for d in dev])
    _assert_equal(r, ref, "device")
    _assert_equal(g.alignBatch(scans), ref, "host")
    # one registration, and an empty batch
    r1 = g.alignBatchDevice([dev[2].data_ptr()], [dev[2].shape[0]])
    _assert_equal(r1, ref[2:3], "one")
    _assert_equal(g.alignBatch(scans[2:3]), ref[2:3], "one host")
    for r0 in (g.alignBatch([]), g.alignBatchDevice([], [])):
        assert r0["pose"].shape == (0, 4, 4) and r0["status"].shape == (0,)


@pytest.mark.gpu
def test_gicp_batch_odd_registrations(b200):
    """Inside one batch: a source with fewer than k = 20 points (its covariances stay zero), a source far from the target
    whose correspondence search finds fewer than 4 pairs (the outer loop breaks at once), and normal scans around them."""
    from lidarslam_ros2_b200 import _capi, synth

    src, tgt, _ = synth.registration_pair("small", 2.0)
    g = _engine(b200, tgt, corr_dist=1.0)
    scans, guesses = _scans_and_guesses(src, 3, seed=5)
    tiny = np.ascontiguousarray(scans[0][::max(1, len(scans[0]) // 12)][:12])
    far = scans[1] + np.array([500.0, -300.0, 40.0], np.float32)
    batch = [scans[0], tiny, scans[1], far, scans[2]]
    bg = [guesses[0], guesses[1], None, guesses[2], guesses[1]]
    bg = [np.eye(4, dtype=np.float32) if x is None else x for x in bg]
    ref = _single(g, batch, bg)
    assert len(tiny) < 20 and ref[3][4] < 4 and ref[3][2] == 0  # the far one: no outer iteration completes
    for slots in (3, 1):
        g.setBatchSlots(slots)
        _assert_equal(g.alignBatch(batch, bg), ref, slots)
    # no target: soft failure like align()
    e = b200.GeneralizedIterativeClosestPoint()
    r = e.alignBatch(scans[:2])
    assert np.all(r["status"] == _capi.ERR_NO_TARGET) and not np.any(r["converged"])


@pytest.mark.gpu
def test_gicp_batch_leaves_handle_source_alone(b200):
    from lidarslam_ros2_b200 import synth

    src, tgt, _ = synth.registration_pair("small", 2.0)
    g = _engine(b200, tgt)
    g.setInputSource(src)
    P0 = g.align()
    cov0 = g.covariances("source")
    m0 = g.numCorrespondences()
    scans, guesses = _scans_and_guesses(src, 4, seed=3)
    g.alignBatch(scans, guesses)
    np.testing.assert_array_equal(g.covariances("source"), cov0)
    P1 = g.align()
    assert np.array_equal(P1, P0) and g.numCorrespondences() == m0


@pytest.mark.gpu
def test_gicp_batch_c3_size(b200):
    """BASELINE config 3 at full size (64-ring scan, ~94k points, against the 1M-point map; corr_dist 5.0, eps 1e-8, k = 20)
    with outer iterations bounded to 6: three perturbed scans in one batch equal their single aligns bitwise (the single
    path's parity with the oracle at this size is test_gicp_parity_baseline_c3_size)."""
    from lidarslam_ros2_b200 import synth

    src, tgt, _ = synth.registration_pair("headline", 2.0)
    g = _engine(b200, tgt)
    g.setTransformationEpsilon(1e-8)
    g.setMaximumIterations(6)
    rng = np.random.default_rng(21)
    scans = [(src[:, :3] + rng.normal(0, 0.003, size=(len(src), 3))).astype(np.float32) for _ in range(3)]
    guesses = [np.eye(4, dtype=np.float32)] * 3
    ref = _single(g, scans, guesses)
    g.setBatchSlots(3)
    _assert_equal(g.alignBatch(scans, guesses), ref, "c3")


def test_gicp_batch_result_layout_matches_ctypes(tmp_path):
    """b200reg_gicp_batch_result as the C compiler lays it out == the ctypes structure the Python mirror reads."""
    import ctypes as C
    import subprocess

    from lidarslam_ros2_b200 import _capi

    fields = [name for name, _ in _capi.GicpBatchResult._fields_]
    src = tmp_path / "layout.c"
    exe = tmp_path / "layout"
    body = "".join(f'  printf("{f} %zu\\n", offsetof(b200reg_gicp_batch_result, {f}));\n' for f in fields)
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "b200reg.h"\nint main(void) {\n'
                   '  printf("sizeof %zu\\n", sizeof(b200reg_gicp_batch_result));\n' + body + "  return 0;\n}\n")
    subprocess.check_call(["cc", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(out["sizeof"]) == C.sizeof(_capi.GicpBatchResult)
    for f in fields:
        assert int(out[f]) == getattr(_capi.GicpBatchResult, f).offset, f
