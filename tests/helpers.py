"""Shared helpers of the parity tests."""
import hashlib
import zlib

import numpy as np

import scenes
from oracle import gut_oracle as go


def oracle_camera(sc, c2w, pose=None):
    pose = scenes.pose7_from_c2w(c2w) if pose is None else pose
    return go.make_camera(sc.width, sc.height, sc.fx, sc.fy, sc.cx, sc.cy, pose, fisheye=getattr(sc, "fisheye", None),
                          ftheta=getattr(sc, "ftheta", None)), pose


def tracer_pose(c2w):
    """The [t, q.xyzw] pose the reference-facing Tracer derives from a float32 T_to_world (tracer.py:404-423)."""
    from threedgut_tracer.tracer import Tracer

    return Tracer._pose_from_c2w(np.asarray(c2w, np.float32))


def oracle_frame(sc, c2w, seed=0, pose=None, with_f64=False):
    """Full oracle forward + backward for one camera; returns a dict of numpy arrays.  with_f64 adds the
    double-precision evaluation of the compositing on the same lists (keys *_64): the tolerance yardstick."""
    cfg = go.default_config()
    cam, pose = oracle_camera(sc, c2w, pose)
    ro, rd = sc.rays()
    pr, bn, rgba, dist, hits = go.forward_all(cfg, cam, ro, rd, sc.particles, sc.sph, sc.sph_degree)
    rng = np.random.default_rng(seed)
    d_rgba = rng.normal(size=rgba.shape).astype(np.float32)
    d_dist = (0.1 * rng.normal(size=dist.shape)).astype(np.float32)
    dp, ds = go.render_backward(cfg, cam, ro, rd, sc.particles, sc.sph, sc.sph_degree, pr, bn, rgba, dist, d_rgba, d_dist)
    out = dict(cfg=cfg, cam=cam, pose=pose, ro=ro, rd=rd, pr=pr, bn=bn, rgba=rgba, dist=dist, hits=hits, d_rgba=d_rgba,
               d_dist=d_dist, dp=dp, ds=ds)
    if with_f64:
        r64, d64, h64 = go.render_forward(cfg, cam, ro, rd, sc.particles, pr, bn, f64=True)
        dp64, ds64 = go.render_backward(cfg, cam, ro, rd, sc.particles, sc.sph, sc.sph_degree, pr, bn, r64, d64, d_rgba, d_dist, f64=True)
        out.update(rgba_64=r64, dist_64=d64, hits_64=h64, dp_64=dp64, ds_64=ds64)
    return out


def image_error_report(name, got, ref, atol=1e-4):
    """(mean abs err, max abs err, number of pixels with any channel off by more than atol)"""
    e = np.abs(np.asarray(got, np.float64) - np.asarray(ref, np.float64)).reshape(ref.shape[0] * ref.shape[1], -1).max(1)
    rep = (float(e.mean()), float(e.max()), int((e > atol).sum()))
    print(f"[parity] {name}: mean|err|={rep[0]:.3e} max|err|={rep[1]:.3e} pixels>{atol:g}: {rep[2]}/{e.size}")
    return rep


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def array_sha(a):
    """SHA-256 of an array's bytes: golden fixtures store this instead of large arrays that must match bit for bit."""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def spread_sample(n, k):
    """min(n, k) distinct indices of range(n), spread over it by a fixed permutation (multiplication by a prime > n), sorted."""
    return np.sort((np.arange(min(n, k), dtype=np.int64) * 2654435761) % n)


def frame_record(f, grad_rows=None):
    """A forward + backward frame reduced to what fits a golden fixture (tests/test_ref_cuda_gpu.py): tile counts, depth, pixels and
    gradient rows on fixed samples; per-tile CRC32 of the sorted value lists; SHA-256 digests of the full integer streams.  `grad_rows`
    defaults to a sample of the particles with a non-zero position / density / rotation / scale gradient."""
    n = f["tiles_count"].shape[0]
    rgba = np.asarray(f["rgba"], np.float32).reshape(-1, 4)
    dist = np.asarray(f["dist"], np.float32).reshape(-1)
    hits = np.asarray(f["hits"], np.float32).reshape(-1)
    dp, ds = np.asarray(f["dp"], np.float32), np.asarray(f["ds"], np.float32)
    if grad_rows is None:
        live = np.flatnonzero(np.any(dp[:, :11] != 0, axis=1))
        grad_rows = live[spread_sample(live.size, 128)]
    ranges, values = np.asarray(f["ranges"], np.int64).reshape(-1, 2), np.asarray(f["sorted_values"], np.uint32)
    pi, di, px, hx = spread_sample(n, 8192), spread_sample(n, 1024), spread_sample(dist.size, 2048), spread_sample(dist.size, 8192)
    return dict(tiles_count=np.asarray(f["tiles_count"], np.uint32)[pi], depth=np.asarray(f["depth"], np.float32)[di],
                tile_crc=np.array([zlib.crc32(values[a:b].tobytes()) for a, b in ranges], np.uint32),
                rgba=rgba[px], dist=dist[px], hits=hits[hx], grad_rows=grad_rows, dp=dp[grad_rows], ds=ds[grad_rows],
                tiles_total=np.int64(np.asarray(f["tiles_count"], np.int64).sum()),
                dist_scale=np.float64(max(1.0, float(np.abs(dist[dist < 1e5]).max()))),
                sha=np.array([f"{k}={array_sha(np.asarray(f[k], t))}" for k, t in (("tiles_count", np.uint32), ("depth", np.float32),
                                                                                    ("sorted_keys", np.uint64), ("sorted_values", np.uint32),
                                                                                    ("ranges", np.uint32))]))


def frac_within(a, b, atol):
    return float(np.mean(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)) <= atol))
