#!/usr/bin/env python
"""Regenerates tests/golden/*.npz from the REFERENCE's own hand-written CUDA math compiled for the host
(oracle/_ref/libgut_ref.so, built from the reference's sources by `make -C oracle ref`, see oracle/ref_gut.cpp):

    python tests/golden/make_golden.py [fixture ...]
    python tests/golden/make_golden.py --gpu     # the reference's own kernels on a GPU (oracle/_ref/libgut_ref_cuda.so, `make -C oracle refcuda`)

The fixtures pin oracle/gut_oracle.c without the reference's sources at hand."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "3dgrut_b200"), os.path.dirname(HERE)):
    sys.path.insert(0, p)

import scenes  # noqa: E402
from helpers import array_sha  # noqa: E402
from oracle import gut_ref as gr  # noqa: E402


def projection():
    sc = scenes.scene_c1(n=300, seed=3, width=96, height=64)
    out = dict(particles=sc.particles, sph=sc.sph, width=sc.width, height=sc.height, fx=sc.fx, fy=sc.fy, cx=sc.cx, cy=sc.cy)
    for i in range(3):
        pose = scenes.pose7_from_c2w(sc.camera(i, 3))
        rf = gr.project(sc.particles, sc.sph, 3, sc.width, sc.height, [sc.fx, sc.fy], [sc.cx, sc.cy], pose, pose)
        keys, vals = gr.expand(sc.width, sc.height, rf["tiles_count"], rf["proj_pos"], rf["conic_opacity"], rf["extent"], rf["depth"])
        view, inv, pos = gr.sensor_matrices(pose, pose)
        out.update({f"pose{i}": pose, f"view{i}": view, f"inv{i}": inv, f"campos{i}": pos, f"keys{i}": keys, f"vals{i}": vals})
        out.update({f"{k}{i}": v for k, v in rf.items()})
    np.savez_compressed(os.path.join(HERE, "gut_projection_ref.npz"), **out)


FISHEYE = (0.05, -0.01, 0.002, -0.0003, 0.33)  # k1..k4, max angle


def projection_fisheye():
    """Same pins through the OpenCV fisheye model (cameraProjections.cuh:120-146).  atan2f comes from the libm of the machine that
    runs this script; the fixture therefore pins the oracle bit for bit only where libm agrees (glibc 2.3x: correctly rounded in
    practice) -- the test accepts a <= 1e-3 fraction of differing tile counts and compares float fields with a 1e-6 tolerance."""
    sc = scenes.scene_c1(n=300, seed=3, width=96, height=64)
    f = 1.2 * sc.width
    out = dict(particles=sc.particles, sph=sc.sph, width=sc.width, height=sc.height, fx=f, fy=f, cx=sc.cx, cy=sc.cy, fisheye=np.asarray(FISHEYE, np.float32))
    gr.set_camera_model(FISHEYE)
    try:
        for i in range(3):
            pose = scenes.pose7_from_c2w(sc.camera(i, 3))
            rf = gr.project(sc.particles, sc.sph, 3, sc.width, sc.height, [f, f], [sc.cx, sc.cy], pose, pose)
            keys, vals = gr.expand(sc.width, sc.height, rf["tiles_count"], rf["proj_pos"], rf["conic_opacity"], rf["extent"], rf["depth"])
            out.update({f"pose{i}": pose, f"keys{i}": keys, f"vals{i}": vals})
            out.update({f"{k}{i}": v for k, v in rf.items() if k != "visibility"})  # undefined for rejected particles in the reference
    finally:
        gr.set_camera_model(None)
    np.savez_compressed(os.path.join(HERE, "gut_projection_fisheye_ref.npz"), **out)


def projection_ftheta():
    """f-theta model (cameraProjections.cuh:148-198), backward polynomial as the reference (Newton inversion)."""
    sc = scenes.scene_c1(n=300, seed=3, width=96, height=64)
    f = 1.2 * sc.width
    a1, a3 = 1.0 / f, 0.04 / f ** 3
    ft = dict(reference_poly=0, bw=[0.0, a1, 0.0, a3, 0.0, 0.0], fw=[0.0, f, 0.0, -0.04 * f, 0.0, 0.0], cde=[1.0, 0.001, -0.002], max_angle=0.36,
              principal=(sc.width / 2.0 - 0.5, sc.height / 2.0 - 0.5))
    out = dict(particles=sc.particles, sph=sc.sph, width=sc.width, height=sc.height, bw=np.asarray(ft["bw"], np.float32),
               fw=np.asarray(ft["fw"], np.float32), cde=np.asarray(ft["cde"], np.float32), max_angle=np.float32(ft["max_angle"]),
               principal=np.asarray(ft["principal"], np.float32))
    gr.set_ftheta(ft)
    try:
        for i in range(3):
            pose = scenes.pose7_from_c2w(sc.camera(i, 3))
            rf = gr.project(sc.particles, sc.sph, 3, sc.width, sc.height, [1.0, 1.0], list(ft["principal"]), pose, pose)
            out.update({f"pose{i}": pose})
            out.update({f"{k}{i}": v for k, v in rf.items() if k != "visibility"})
    finally:
        gr.set_camera_model(None)
    np.savez_compressed(os.path.join(HERE, "gut_projection_ftheta_ref.npz"), **out)


def hits():
    rng = np.random.default_rng(2024)
    rows = []
    for degree in (2, 4):
        for _ in range(300):
            pos = rng.normal(size=3) * 0.3
            scl = np.exp(rng.normal(np.log(0.2), 0.5, 3))
            q = rng.normal(size=4)
            q /= np.linalg.norm(q)
            p = np.concatenate([pos, [rng.uniform(0.02, 1.0)], q, scl, [0]]).astype(np.float32)
            ro = np.array([0, 0, -3], np.float32) + rng.normal(size=3).astype(np.float32) * 0.1
            rd = pos + rng.normal(size=3) * 0.25 - ro
            rd = (rd / np.linalg.norm(rd)).astype(np.float32)
            rgb = rng.uniform(0, 1, 3).astype(np.float32)
            T, C0, D = np.float32(rng.uniform(0.05, 1)), rng.uniform(0, 0.5, 3).astype(np.float32), np.float32(rng.uniform(0, 2))
            Tint, Cint, Dint = np.float32(T * rng.uniform(0.001, 0.9)), (C0 + rng.uniform(0.1, 1, 3)).astype(np.float32), np.float32(D + rng.uniform(0.1, 3))
            Tg, Cg, Dg = np.float32(rng.normal()), rng.normal(size=3).astype(np.float32), np.float32(rng.normal())
            acc, T1, C1, D1 = gr.hit_fwd(degree, ro, rd, p, rgb, float(T), C0, float(D))
            g, rg, Tb, Cb, Db = gr.hit_bwd(degree, ro, rd, p, rgb, 1e-4, float(Tint), float(T), float(Tg), Cint, C0, Cg, float(Dint), float(D), float(Dg))
            rows.append(np.concatenate([[degree], p, ro, rd, rgb, [T], C0, [D], [Tint], Cint, [Dint], [Tg], Cg, [Dg],
                                        [acc, T1], C1, [D1], g, rg, [Tb], Cb, [Db]]).astype(np.float64))
    np.savez_compressed(os.path.join(HERE, "gut_hits_ref.npz"), rows=np.stack(rows))


def sph():
    rng = np.random.default_rng(9)
    c = rng.normal(size=(64, 48)).astype(np.float32)
    d = rng.normal(size=(64, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    out = np.stack([np.stack([gr.sph(deg, c[i], d[i], clamped=False) for i in range(64)]) for deg in range(4)])
    np.savez_compressed(os.path.join(HERE, "gut_sph_ref.npz"), coeffs=c, dirs=d, rgb=out)


def _digests(out, case, arrays):
    out[f"{case}__sha"] = np.array([f"{k}={array_sha(v)}" for k, v in arrays.items()])


def _projection_record(out, case, rf, keys, vals):
    """What tests/test_oracle_vs_ref.py compares bit for bit, as SHA-256 digests (tile counts and visibility in full)."""
    out[f"{case}__tiles_count"] = rf["tiles_count"]
    out[f"{case}__visibility"] = rf["visibility"].astype(np.int8)
    order = np.argsort(keys, kind="stable")
    _digests(out, case, dict({k: rf[k] for k in ("depth", "proj_pos", "conic_opacity", "extent")}, rgb_visible=rf["rgb"][rf["tiles_count"] > 0],
                             keys=keys, vals=vals, sorted_keys=keys[order], sorted_vals=vals[order]))


def ref_cases():
    """The reference's side of every case of tests/test_oracle_vs_ref.py, on the same inputs (gut_ref_cases.npz)."""
    import test_oracle_vs_ref as t

    out = {}
    sc = scenes.scene_c1(bands=True)
    for i in range(6):
        pose = scenes.pose7_from_c2w(sc.camera(i, 6))
        rf = gr.project(sc.particles, sc.sph, 3, sc.width, sc.height, [sc.fx, sc.fy], [sc.cx, sc.cy], pose, pose)
        keys, vals = gr.expand(sc.width, sc.height, rf["tiles_count"], rf["proj_pos"], rf["conic_opacity"], rf["extent"], rf["depth"])
        _projection_record(out, f"pinhole{i}", rf, keys, vals)
    f = 1.2 * sc.width
    gr.set_camera_model(t.FISHEYE)
    try:
        for i in range(4):
            pose = scenes.pose7_from_c2w(sc.camera(i, 4))
            rf = gr.project(sc.particles, sc.sph, 3, sc.width, sc.height, [f, f], [sc.cx, sc.cy], pose, pose)
            keys, vals = gr.expand(sc.width, sc.height, rf["tiles_count"], rf["proj_pos"], rf["conic_opacity"], rf["extent"], rf["depth"])
            _projection_record(out, f"fisheye{i}", rf, keys, vals)
    finally:
        gr.set_camera_model(None)
    for poly in (0, 1):
        ft = t._ftheta(sc.width, sc.height, poly)
        gr.set_ftheta(ft)
        try:
            for i in range(3):
                pose = scenes.pose7_from_c2w(sc.camera(i, 3))
                rf = gr.project(sc.particles, sc.sph, 3, sc.width, sc.height, [1.0, 1.0], list(ft["principal"]), pose, pose)
                keys, vals = gr.expand(sc.width, sc.height, rf["tiles_count"], rf["proj_pos"], rf["conic_opacity"], rf["extent"], rf["depth"])
                _projection_record(out, f"ftheta{poly}_{i}", rf, keys, vals)
        finally:
            gr.set_camera_model(None)
    p0 = scenes.pose7_from_c2w(sc.camera(1, 40))
    p1 = scenes.pose7_from_c2w(sc.camera(2, 40))
    for model in ("pinhole", "fisheye"):
        fe = t.FISHEYE if model == "fisheye" else None
        f = 1.2 * sc.width if model == "fisheye" else sc.fx
        for kind in (1, 2, 3, 4):
            gr.set_camera_model(fe)
            gr.set_rolling_shutter(kind)
            try:
                rf = gr.project(sc.particles, sc.sph, 3, sc.width, sc.height, [f, f], [sc.cx, sc.cy], p0, p1)
            finally:
                gr.set_rolling_shutter(0)
                gr.set_camera_model(None)
            case = f"shutter_{model}{kind}"
            out[f"{case}__tiles_count"] = rf["tiles_count"]
            _digests(out, case, {k: rf[k] for k in ("depth", "proj_pos", "conic_opacity", "extent")})
    sc8 = scenes.scene_c1()
    for i in range(8):
        pose = scenes.pose7_from_c2w(sc8.camera(i, 8))
        for k, v in zip(("view", "inv", "pos"), gr.sensor_matrices(pose, pose)):
            out[f"sensor{i}__{k}"] = v
    for degree in (2, 4):
        # the same random stream as the test; only accepted hits carry values (a rejected one is compared by its flag)
        rng = np.random.default_rng(degree)
        acc_all, rows = [], []
        for _ in range(1500):
            p, ro, rd = t._random_hit_case(rng)
            rgb = rng.uniform(0, 1, 3).astype(np.float32)
            T, C0, D = float(rng.uniform(0.05, 1)), rng.uniform(0, 0.5, 3).astype(np.float32), float(rng.uniform(0, 2))
            acc, T1, _, D1 = gr.hit_fwd(degree, ro, rd, p, rgb, T, C0, D)
            Tint, Cint, Dint = T * rng.uniform(0.001, 0.9), C0 + rng.uniform(0.1, 1, 3).astype(np.float32), D + rng.uniform(0.1, 3)
            Tg, Cg, Dg = float(rng.normal()), rng.normal(size=3).astype(np.float32), float(rng.normal())
            g, rg, Tb, _, _ = gr.hit_bwd(degree, ro, rd, p, rgb, 1e-4, Tint, T, Tg, Cint, C0, Cg, Dint, D, Dg)
            acc_all.append(acc)
            if acc:
                rows.append(np.concatenate([[T1, D1], g[:11], rg, [Tb]]))
        out[f"hits{degree}__accepted"] = np.asarray(acc_all, np.int8)
        out[f"hits{degree}__rows"] = np.asarray(rows, np.float32)  # T after, D after, d particle[:11], d rgb, T adjoint
    rng = np.random.default_rng(5)
    sph_out = []
    for deg in range(4):
        for _ in range(50):
            c = rng.normal(size=48).astype(np.float32)
            d = rng.normal(size=3)
            d = (d / np.linalg.norm(d)).astype(np.float32)
            sph_out.append(gr.sph(deg, c, d, clamped=False))
    out["sph__rgb"] = np.stack(sph_out)
    np.savez_compressed(os.path.join(HERE, "gut_ref_cases.npz"), **out)


def _run_reference_gpu(sc, pose, d_rgba, d_dist):
    """One forward + backward frame through the reference's own 3DGUT kernels (oracle/_ref/libgut_ref_cuda.so) on cuda:0."""
    import torch

    from oracle import gut_ref_cuda as grc

    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    ro, rd = sc.rays()
    particles, sph, tro, trd = t(sc.particles), t(sc.sph), t(ro), t(rd)
    rr = grc.ReferenceRaster()
    s = torch.cuda.current_stream(dev).cuda_stream
    rgba, dist, hits, vis = rr.trace(torch, s, 0, sc.sph_degree, particles, sph, sc.width, sc.height, sc.fx, sc.fy, sc.cx, sc.cy, pose, tro, trd)
    torch.cuda.synchronize()
    tiles = ((sc.width + 15) // 16) * ((sc.height + 15) // 16)
    dbg = {k: rr.debug(k, sc.n, tiles) for k in ("tiles_count", "sorted_keys", "sorted_values", "ranges", "depth")}
    dp, ds = rr.trace_bwd(torch, s, 0, sc.sph_degree, particles, sph, sc.width, sc.height, sc.fx, sc.fy, sc.cx, sc.cy, pose, tro, trd, rgba,
                          t(d_rgba), dist, t(d_dist))
    torch.cuda.synchronize()
    out = dict(rgba=rgba.cpu().numpy(), dist=dist.cpu().numpy(), hits=hits.cpu().numpy(), dp=dp.cpu().numpy(), ds=ds.cpu().numpy(), **dbg)
    rr.close()
    return out


def ref_gpu():
    """The reference's GPU frames of tests/test_ref_cuda_gpu.py, reduced by helpers.frame_record (ref_gpu_<case>.npz).  Needs a GPU."""
    import test_ref_cuda_gpu as t
    from helpers import frame_record

    for case, (make_scene, cam_index, n_cams) in t.CASES.items():
        sc = make_scene()
        _, pose, d_rgba, d_dist = t.frame_inputs(sc, cam_index, n_cams)
        np.savez_compressed(os.path.join(HERE, f"ref_gpu_{case}.npz"), **frame_record(_run_reference_gpu(sc, pose, d_rgba, d_dist)))


CPU_FIXTURES = dict(projection=projection, projection_fisheye=projection_fisheye, projection_ftheta=projection_ftheta, hits=hits, sph=sph,
                    ref_cases=ref_cases)

if __name__ == "__main__":
    if sys.argv[1:] == ["--gpu"]:
        ref_gpu()
    else:
        assert gr.available(), "oracle/_ref could not be built (needs the reference sources, see oracle/Makefile)"
        for name in sys.argv[1:] or list(CPU_FIXTURES):
            CPU_FIXTURES[name]()
    print("golden fixtures written to", HERE)
