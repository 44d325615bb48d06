"""Parity against the REFERENCE'S OWN 3DGUT kernels running on the GPU: oracle/_ref/libgut_ref_cuda.so is threedgut_tracer/src/gutRenderer.cu
(projectOnTiles, CUB scan, expandTileProjections, 44-bit CUB radix sort, tile ranges, render, renderBackward with the hand-written adjoint,
projectBackward, and the host orchestration around them) compiled UNMODIFIED for sm_100a in the build container, with only the slangc output
replaced by a hand translation (oracle/ref_cuda/threedgutSlang.cuh).  This is the pin the round-1 oracle lacked: the CPU oracle and the
product are both compared with what the reference's kernels compute on identical tensors.

The reference binary is built the way its setup script builds it (-use_fast_math -O3: FMA contraction, approximate div / sqrt / exp), ours
keeps the projection stage IEEE (DESIGN.md section 3), so integers are compared as "equal except for a counted borderline set":
  tile counts equal on >= 99.9 % of the particles, and wherever they are equal for ALL particles of a tile list the sorted (key, value)
  stream is bit-identical; RGBA / dist mean |diff| <= 1e-5, outliers as in the other parity tests; gradients rel-L2 <= 3e-3 against the
  reference (two fast-math evaluations of a discontinuous accept test; the oracle-vs-reference figure is printed beside ours).
First run on a B200 (profiles/r02_f_reference_kernels_on_gpu.md): C1 tile counts equal on 100 %, all 64 tile lists identical in order; C2
tile counts equal on 99.9983-99.9993 % of 300k particles, 2478-2482 of 2500 tile lists identical in order (the reference's -use_fast_math
build contracts the depth FMA: 3.4 % of the depth keys differ in the last bit, which reorders neighbours with near-equal depth), images
35-56 of 640 000 pixels off by more than 1e-4, gradients 2e-5 .. 6e-4 -- except d_quat of C2 camera 41 at 2.22e-3, the frame and tensor
whose fp32-vs-fp64 yardstick is 2.24e-3 (one borderline anisotropic particle, tests/test_gut_headline_parity_gpu.py): hence 3e-3 here.

The reference's frames are stored in tests/golden/ref_gpu_<case>.npz (written on a B200 by `tests/golden/make_golden.py --gpu`), reduced
by helpers.frame_record: tile counts, depth, pixels and gradient rows on fixed samples, a CRC32 per tile list, digests of the full integer
streams.  Every figure below is taken over those samples, with the thresholds of the full-frame comparison."""
import os

import numpy as np
import pytest

import scenes
from helpers import frame_record, image_error_report, oracle_frame, rel_l2, tracer_pose

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# case -> (scene, camera index, cameras on the orbit)
CASES = {
    "c1_cam1": (lambda: scenes.scene_c1(), 1, 8),
    "c1-dc_cam5": (lambda: scenes.scene_c1(bands=False), 5, 8),
    "c2_cam3": (lambda: scenes.scene_c2(), 3, 100),
    "c2_cam41": (lambda: scenes.scene_c2(), 41, 100),
    "c3-400k_cam2": (lambda: scenes.scene_c3(n=400_000), 2, 16),
}


def frame_inputs(sc, cam_index, n_cams):
    c2w = sc.camera(cam_index, n_cams)
    rng = np.random.default_rng(cam_index)
    d_rgba = rng.normal(size=(sc.height, sc.width, 4)).astype(np.float32)
    d_dist = (0.1 * rng.normal(size=(sc.height, sc.width, 1))).astype(np.float32)
    return c2w, tracer_pose(c2w), d_rgba, d_dist


def _load_record(case):
    z = np.load(os.path.join(GOLDEN, f"ref_gpu_{case}.npz"))
    return {k: z[k] for k in z.files}


def _digests(rec):
    return dict(v.split("=") for v in rec.pop("sha"))


def _run_ours(sc, pose, d_rgba, d_dist):
    import b200_native as nat

    ctx = nat.Context(nat.default_config(), 0)
    cam = nat.Camera()
    cam.width, cam.height = sc.width, sc.height
    cam.principal[:] = [sc.cx, sc.cy]
    cam.focal[:] = [sc.fx, sc.fy]
    cam.pose_start[:] = [float(v) for v in pose]
    cam.pose_end[:] = [float(v) for v in pose]
    n, hw = sc.n, sc.width * sc.height
    rgba, dist, hits, vis = (np.zeros((hw, 4), np.float32), np.zeros(hw, np.float32), np.zeros(hw, np.float32), np.zeros(n, np.float32))
    p = lambda a: a.ctypes.data  # noqa: E731
    ro, rd = sc.rays()
    ro, rd = np.ascontiguousarray(ro), np.ascontiguousarray(rd)
    ctx.forward_host(cam, n, p(sc.particles), p(sc.sph), sc.sph_degree, p(ro), p(rd), p(rgba), p(dist), p(hits), p(vis))
    dbg = dict(tiles_count=ctx.debug_copy(nat.DBG_TILES_COUNT), sorted_keys=ctx.debug_copy(nat.DBG_SORTED_KEYS),
               sorted_values=ctx.debug_copy(nat.DBG_SORTED_VALUES), ranges=ctx.debug_copy(nat.DBG_TILE_RANGES), depth=ctx.debug_copy(nat.DBG_DEPTH))
    dp, ds = np.zeros((n, 12), np.float32), np.zeros((n, 48), np.float32)
    d_rgba, d_dist = np.ascontiguousarray(d_rgba), np.ascontiguousarray(d_dist)
    ctx.backward_host(cam, n, p(sc.particles), p(sc.sph), sc.sph_degree, p(ro), p(rd), p(rgba), p(d_rgba), p(dist), p(d_dist), p(dp), p(ds))
    ctx.close()
    return dict(rgba=rgba.reshape(sc.height, sc.width, 4), dist=dist.reshape(sc.height, sc.width, 1), hits=hits.reshape(sc.height, sc.width, 1),
                vis=vis.view(np.int32), dp=dp, ds=ds, **dbg)


def _compare(case, with_oracle):
    make_scene, cam_index, n_cams = CASES[case]
    sc = make_scene()
    label = case.split("_cam")[0]
    ref = _load_record(case)
    ref_sha = _digests(ref)
    c2w, pose, d_rgba, d_dist = frame_inputs(sc, cam_index, n_cams)
    arms = {"ours": _run_ours(sc, pose, d_rgba, d_dist)}
    if with_oracle:
        o = oracle_frame(sc, c2w, seed=cam_index, pose=pose)
        arms["oracle"] = dict(rgba=o["rgba"], dist=o["dist"], hits=o["hits"], dp=o["dp"], ds=o["ds"], tiles_count=o["pr"].tiles_count,
                              sorted_keys=o["bn"].sorted_keys, sorted_values=o["bn"].sorted_values, ranges=o["bn"].ranges, depth=o["pr"].depth)
        assert np.array_equal(o["d_rgba"], d_rgba) and np.array_equal(o["d_dist"], d_dist)
    P = ref["rgba"].shape[0]  # sampled pixels
    cols = dict(pos=slice(0, 3), dns=slice(3, 4), quat=slice(4, 8), scl=slice(8, 11))
    for name, full in arms.items():
        a = frame_record(full, ref["grad_rows"])
        a_sha = _digests(a)
        tc_same = float(np.mean(a["tiles_count"] == ref["tiles_count"]))
        depth_same = float(np.mean(a["depth"].view(np.uint32) == ref["depth"].view(np.uint32)))
        print(f"[ref-gpu] {label} cam{cam_index} {name}: tile counts equal on {tc_same * 100:.4f} % of {a['tiles_count'].size} sampled particles "
              f"(I {int(a['tiles_total'])} vs reference {int(ref['tiles_total'])}), depth bits equal on {depth_same * 100:.4f} % of a sample")
        assert tc_same >= 0.999
        if a_sha["tiles_count"] == ref_sha["tiles_count"] and a_sha["depth"] == ref_sha["depth"]:
            assert a_sha["sorted_keys"] == ref_sha["sorted_keys"] and a_sha["sorted_values"] == ref_sha["sorted_values"]
            assert a_sha["ranges"] == ref_sha["ranges"]
            print(f"[ref-gpu] {label} cam{cam_index} {name}: sorted (key, value) stream and tile ranges BIT-IDENTICAL to the reference's CUB 44-bit sort")
        else:
            # per tile: the particle lists (order included) must agree except where a tile count differed
            T = ref["tile_crc"].shape[0]
            same_tiles = int(np.sum(a["tile_crc"] == ref["tile_crc"]))
            print(f"[ref-gpu] {label} cam{cam_index} {name}: {same_tiles}/{T} tile lists identical (order included)")
            assert same_tiles >= 0.97 * T
        mean_e, max_e, bad = image_error_report(f"{label} cam{cam_index} {name} vs reference-gpu rgba", a["rgba"][:, None], ref["rgba"][:, None])
        assert mean_e <= 1e-5 and max_e <= 5e-2 and bad <= max(3, int(4e-4 * P))
        dscale = float(ref["dist_scale"])
        mean_e, _, bad = image_error_report(f"{label} cam{cam_index} {name} vs reference-gpu dist", a["dist"][:, None, None], ref["dist"][:, None, None],
                                            atol=1e-4 * dscale)
        assert mean_e <= 1e-5 * dscale and bad <= max(3, int(4e-4 * P))
        same_hits = float(np.mean(a["hits"] == ref["hits"]))
        errs = {k: rel_l2(a["dp"][:, v], ref["dp"][:, v]) for k, v in cols.items()}
        errs["sph"] = rel_l2(a["ds"], ref["ds"])
        print(f"[ref-gpu] {label} cam{cam_index} {name}: hit counts equal on {same_hits * 100:.4f} % of {a['hits'].size} sampled pixels; "
              f"gradient rel-L2 vs reference-gpu over {ref['grad_rows'].size} sampled particles:", {k: f"{v:.2e}" for k, v in errs.items()})
        assert same_hits >= 0.999
        for k, v in errs.items():
            assert v <= 3e-3, (name, k, v)


def test_c1_reference_kernels_vs_oracle_and_ours():
    """C1 (1k Gaussians, 128x128): CPU oracle AND product against the reference's kernels."""
    _compare("c1_cam1", with_oracle=True)


def test_c1_dc_only_reference_kernels():
    _compare("c1-dc_cam5", with_oracle=True)


@pytest.mark.parametrize("cam_index", [3, 41])
def test_c2_reference_kernels_vs_oracle_and_ours(cam_index):
    """BASELINE configs[1] at full scale (300k Gaussians, 800x800): product and oracle against the reference's kernels."""
    _compare(f"c2_cam{cam_index}", with_oracle=True)


def test_c3_like_reference_kernels_vs_ours():
    _compare("c3-400k_cam2", with_oracle=False)
