"""Pins the C restatement (oracle/gut_oracle.c) against the REFERENCE's own hand-written CUDA math compiled for
the host (oracle/_ref/libgut_ref.so, oracle/ref_gut.cpp).  The reference's results on exactly these inputs are stored in
tests/golden/gut_ref_cases.npz (tests/golden/make_golden.py ref_cases): arrays compared bit for bit are kept as SHA-256
digests, tile counts and visibility in full, single-hit results as values."""
import os

import numpy as np
import pytest

import scenes
from helpers import array_sha
from oracle import gut_oracle as go

_Z = None


def _ref(case):
    """The reference's stored results of one case: {name: array}."""
    global _Z
    if _Z is None:
        _Z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gut_ref_cases.npz"))
    out = {}
    for k in _Z.files:
        if k.startswith(case + "__"):
            name = k.split("__", 1)[1]
            if name == "sha":
                out.update(v.split("=") for v in _Z[k])
            else:
                out[name] = _Z[k]
    return out


def _same(a, digest):
    return array_sha(a) == digest


def _cam(sc, i, n=6):
    pose = scenes.pose7_from_c2w(sc.camera(i, n))
    return go.make_camera(sc.width, sc.height, sc.fx, sc.fy, sc.cx, sc.cy, pose), pose


@pytest.mark.parametrize("cam_index", range(6))
def test_projection_and_keys_bit_identical(cam_index):
    sc = scenes.scene_c1(bands=True)
    cfg = go.default_config()
    cam, pose = _cam(sc, cam_index)
    pr = go.project(cfg, cam, sc.particles, sc.sph, 3)
    rf = _ref(f"pinhole{cam_index}")
    assert pr.tiles_count.sum() > 1000
    assert np.array_equal(pr.tiles_count, rf["tiles_count"])
    for k in ("depth", "proj_pos", "conic_opacity", "extent"):
        assert _same(getattr(pr, k), rf[k]), k
    vis = pr.tiles_count > 0
    assert _same(pr.rgb[vis], rf["rgb_visible"])
    # visibility: identical wherever the reference's value is defined (it reads an uninitialised covariance when the
    # projection was rejected, gutProjector.cuh:245-275)
    differs = pr.visibility != rf["visibility"]
    assert not np.any(differs & (pr.visibility == 1))
    bn = go.bin_tiles(cfg, cam, pr)
    assert _same(bn.unsorted_keys, rf["keys"]) and _same(bn.unsorted_values, rf["vals"])
    # the reference's expanded keys in a stable 64-bit sort (tile bits are the high bits: a full sort == the masked one)
    assert _same(bn.sorted_keys, rf["sorted_keys"]) and _same(bn.sorted_values, rf["sorted_vals"])


FISHEYE = (0.05, -0.01, 0.002, -0.0003, 0.33)  # k1..k4, max angle (rad): some particles fall outside the valid cone


@pytest.mark.parametrize("cam_index", range(4))
def test_fisheye_projection_bit_identical(cam_index):
    """OpenCV fisheye model (cameraProjections.cuh:120-146) through the whole projection + key expansion: bit-identical with the
    reference's own code compiled for the host (both sides call the same libm atan2f)."""
    sc = scenes.scene_c1(bands=True)
    cfg = go.default_config()
    pose = scenes.pose7_from_c2w(sc.camera(cam_index, 4))
    f = 1.2 * sc.width  # fisheye focal: pixels per radian (the image spans about +-0.4 rad, the valid cone 0.33)
    cam = go.make_camera(sc.width, sc.height, f, f, sc.cx, sc.cy, pose, fisheye=FISHEYE)
    pr = go.project(cfg, cam, sc.particles, sc.sph, 3)
    rf = _ref(f"fisheye{cam_index}")
    assert pr.tiles_count.sum() > 500
    assert (pr.tiles_count == 0).sum() > 0  # the max-angle / resolution rejections are exercised
    assert np.array_equal(pr.tiles_count, rf["tiles_count"])
    for k in ("depth", "proj_pos", "conic_opacity", "extent"):
        assert _same(getattr(pr, k), rf[k]), k
    bn = go.bin_tiles(cfg, cam, pr)
    assert _same(bn.unsorted_keys, rf["keys"]) and _same(bn.unsorted_values, rf["vals"])
    # and it differs from the pinhole projection of the same scene (the model switch is really taken)
    pin = go.project(cfg, go.make_camera(sc.width, sc.height, f, f, sc.cx, sc.cy, pose), sc.particles, sc.sph, 3)
    assert not np.array_equal(pin.proj_pos, pr.proj_pos)


def _ftheta(width, height, reference_poly):
    """equidistant-like f-theta camera: backward polynomial theta = a1 r + a3 r^3, forward its low-order inverse"""
    f = 1.2 * width
    a1, a3 = 1.0 / f, 0.04 / f ** 3
    return dict(reference_poly=reference_poly, bw=[0.0, a1, 0.0, a3, 0.0, 0.0], fw=[0.0, f, 0.0, -0.04 * f, 0.0, 0.0], cde=[1.0, 0.001, -0.002],
                max_angle=0.36, principal=(width / 2.0 - 0.5, height / 2.0 - 0.5))


@pytest.mark.parametrize("reference_poly", [0, 1])
@pytest.mark.parametrize("cam_index", range(3))
def test_ftheta_projection_bit_identical(cam_index, reference_poly):
    """f-theta model (cameraProjections.cuh:148-198), both reference polynomials (Newton inversion of the backward polynomial /
    direct forward polynomial), through projection + key expansion: bit-identical with the reference's code compiled for the host."""
    sc = scenes.scene_c1(bands=True)
    cfg = go.default_config()
    pose = scenes.pose7_from_c2w(sc.camera(cam_index, 3))
    ft = _ftheta(sc.width, sc.height, reference_poly)
    cam = go.make_camera(sc.width, sc.height, 1.0, 1.0, 0.0, 0.0, pose, ftheta=ft)
    pr = go.project(cfg, cam, sc.particles, sc.sph, 3)
    rf = _ref(f"ftheta{reference_poly}_{cam_index}")
    assert pr.tiles_count.sum() > 500 and (pr.tiles_count == 0).sum() > 0
    assert np.array_equal(pr.tiles_count, rf["tiles_count"])
    for k in ("proj_pos", "conic_opacity", "extent"):
        assert _same(getattr(pr, k), rf[k]), k
    bn = go.bin_tiles(cfg, cam, pr)
    assert _same(bn.unsorted_keys, rf["keys"]) and _same(bn.unsorted_values, rf["vals"])


@pytest.mark.parametrize("kind", [1, 2, 3, 4])
@pytest.mark.parametrize("model", ["pinhole", "fisheye"])
def test_rolling_shutter_projection_bit_identical(kind, model):
    """projectPointWithShutter (cameraProjections.cuh:218-257) with a sensor that moves and rotates during the exposure: 5 iterations of
    pose(time of the projected row / column) -> projection, for the four readout directions."""
    sc = scenes.scene_c1(bands=True)
    cfg = go.default_config()
    p0 = scenes.pose7_from_c2w(sc.camera(1, 40))
    p1 = scenes.pose7_from_c2w(sc.camera(2, 40))  # 9 degrees further along the orbit
    fe = FISHEYE if model == "fisheye" else None
    f = 1.2 * sc.width if model == "fisheye" else sc.fx
    cam = go.make_camera(sc.width, sc.height, f, f, sc.cx, sc.cy, p0, p1, fisheye=fe, rolling_shutter=kind)
    pr = go.project(cfg, cam, sc.particles, sc.sph, 3)
    rf = _ref(f"shutter_{model}{kind}")
    assert pr.tiles_count.sum() > 500
    assert np.array_equal(pr.tiles_count, rf["tiles_count"])
    for k in ("depth", "proj_pos", "conic_opacity", "extent"):
        assert _same(getattr(pr, k), rf[k]), k
    # the shutter really matters: the global-shutter projection of the same poses differs
    glob = go.project(cfg, go.make_camera(sc.width, sc.height, f, f, sc.cx, sc.cy, p0, p1, fisheye=fe), sc.particles, sc.sph, 3)
    assert not np.array_equal(glob.proj_pos, pr.proj_pos)


def test_sensor_pose_maths_identical():
    sc = scenes.scene_c1()
    for i in range(8):
        cam, pose = _cam(sc, i, 8)
        a = go.sensor_matrices(cam)
        rf = _ref(f"sensor{i}")
        for x, k in zip(a, ("view", "inv", "pos")):
            assert np.array_equal(x, rf[k]), k


def _random_hit_case(rng):
    pos = rng.normal(size=3) * 0.3
    scl = np.exp(rng.normal(np.log(0.2), 0.5, 3))
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    p = np.concatenate([pos, [rng.uniform(0.02, 1.0)], q, scl, [0]]).astype(np.float32)
    ro = np.array([0, 0, -3], np.float32) + rng.normal(size=3).astype(np.float32) * 0.1
    rd = pos + rng.normal(size=3) * 0.25 - ro
    rd = (rd / np.linalg.norm(rd)).astype(np.float32)
    return p, ro, rd


@pytest.mark.parametrize("degree", [2, 4])
def test_single_hit_forward_and_adjoint_match_reference(degree):
    rng = np.random.default_rng(degree)
    cfg = go.default_config()
    cfg.kernel_degree = degree
    rf = _ref(f"hits{degree}")
    ref_rows = iter(rf["rows"])  # per accepted hit: T after, D after, d particle[:11], d rgb, T adjoint
    accepted, worst = 0, 0.0
    for acc_ref in rf["accepted"]:
        p, ro, rd = _random_hit_case(rng)
        rgb = rng.uniform(0, 1, 3).astype(np.float32)
        T, C0, D = float(rng.uniform(0.05, 1)), rng.uniform(0, 0.5, 3).astype(np.float32), float(rng.uniform(0, 2))
        acc, alpha, t = go.hit_forward(cfg, ro, rd, p)
        assert acc == acc_ref
        if acc:
            row = next(ref_rows)
            T_ref, D_ref, g_ref, rg_ref, Tb_ref = row[0], row[1], row[2:13], row[13:16], row[16]
            w = np.float32(alpha) * np.float32(T)
            assert abs(np.float32(T) * (np.float32(1) - np.float32(alpha)) - T_ref) <= 1e-6
            assert abs(np.float32(D) + np.float32(t) * w - D_ref) <= 1e-5 * max(1.0, abs(D_ref))
        Tint, Cint, Dint = T * rng.uniform(0.001, 0.9), C0 + rng.uniform(0.1, 1, 3).astype(np.float32), D + rng.uniform(0.1, 3)
        Tg, Cg, Dg = float(rng.normal()), rng.normal(size=3).astype(np.float32), float(rng.normal())
        acc2, g, rg, Tb, _, _ = go.hit_backward(cfg, ro, rd, p, rgb, Tint, T, Tg, Cint, C0, Cg, Dint, D, Dg)
        assert acc2 == acc
        if acc:
            accepted += 1
            worst = max(worst, float(np.abs(g_ref - g).max() / (np.abs(g_ref).max() + 1e-12)), float(np.abs(rg_ref - rg).max()))
            assert abs(Tb - Tb_ref) <= 1e-6
    assert accepted > 500 and accepted == len(rf["rows"])
    assert worst <= 5e-5


def test_sph_eval_and_coefficient_adjoint_match_reference():
    rng = np.random.default_rng(5)
    want = iter(_ref("sph")["rgb"])
    for deg in range(4):
        for _ in range(50):
            c = rng.normal(size=48).astype(np.float32)
            d = rng.normal(size=3)
            d = (d / np.linalg.norm(d)).astype(np.float32)
            assert np.array_equal(go.sph_eval(deg, c, d), next(want))
