"""Count the raster kernel's (tile, triangle) work on the CPU: seeded states of a scenario (the oracle's levels and cameras), the
triangle set-up restated in numpy (vertex stage, near / far clipping, back-face test, 8-bit sub-pixel snap, pixel box, edge constants
with the top-left bias), then per view and 32x4 tile:

  list      triangles in the view's list (front-facing, covering a pixel centre of the viewport)
  box       (tile, triangle) pairs whose pixel box overlaps the tile      -- what a per-tile scan of the list hands to the warp
  kept      pairs the kernel's conservative bin test keeps (every edge at the tile sample where it is largest, exact integers)
  covered   pairs that cover at least one sample of the tile
  small     covered pairs that cover at most 4 samples of the tile

The vertex stage is float32 numpy, not the kernel's exact operation order, so a vertex may snap one sub-pixel apart now and then: the
counts are for sizing work, not for checking frames.

  python tools/tile_pairs.py --scenario Collect --envs 1024 --agents 4 [--steps 0] [--views 512]
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import orc  # noqa: E402

F32 = np.float32


def projection(w, h):
    aspect = F32(w) / F32(h)
    half_tan = F32(np.tan(np.float64(F32(100.0) * F32(0.01745329251994329576923690768489)) / 2.0))
    near, far = F32(0.01), F32(120.0)
    return F32(1.0) / half_tan, -aspect / half_tan, far / (near - far), far * near / (near - far)


MESHES = {}


def mesh(kind):
    if kind not in MESHES:
        vtx, idx = orc.mesh(kind)
        MESHES[kind] = (vtx.view(np.float32).reshape(-1, 6)[:, :3].copy(), idx.reshape(-1, 3).astype(np.int64))
    return MESHES[kind]


def clip_near_far(tri):
    poly = [tri[k] for k in range(3)]
    for plane in (0, 1):
        dist = (lambda c: c[2]) if plane == 0 else (lambda c: c[3] - c[2])
        out = []
        for i in range(len(poly)):
            a, b = poly[i], poly[(i + 1) % len(poly)]
            da, db = dist(a), dist(b)
            if da >= 0:
                out.append(a)
            if (da >= 0) != (db >= 0):
                out.append(a + (da / (da - db)) * (b - a) if da >= 0 else b + (db / (db - da)) * (a - b))
        poly = out
        if len(poly) < 3:
            return []
    return [np.array([poly[0], poly[k], poly[k + 1]]) for k in range(1, len(poly) - 1)]


def view_triangles(view16, inst, w, h, proj):
    """clip-space triangles (T, 3, 4) float64 of one view, in draw order"""
    p00, p11, p22, p32 = proj
    V = view16.reshape(4, 4).T.astype(F32)  # row-major view matrix
    out = []
    for kind in range(5):
        rows = inst[inst[:, 0] == kind]
        if not len(rows):
            continue
        verts, tris = mesh(kind)
        M = rows[:, 2:18].reshape(-1, 4, 4).transpose(0, 2, 1).astype(F32)  # row-major model matrices
        MV = np.einsum("ij,njk->nik", V, M).astype(F32)
        vh = np.concatenate([verts, np.ones((len(verts), 1), F32)], axis=1)
        cam = np.einsum("nij,vj->nvi", MV[:, :3, :], vh).astype(F32)
        clip = np.stack([cam[..., 0] * p00, cam[..., 1] * p11, cam[..., 2] * p22 + p32, -cam[..., 2]], axis=-1).astype(np.float64)
        out.append(clip[:, tris].reshape(-1, 3, 4))
    return np.concatenate(out) if out else np.zeros((0, 3, 4))


def setup(clip, w, h):
    """snapped screen triangles -> (A, B, C, box) of the front-facing ones that cover a pixel centre (kernel: triBox + writeTri)"""
    needs = ((clip[:, :, 2] < 0) | (clip[:, :, 3] - clip[:, :, 2] < 0)).any(axis=1)
    side = np.zeros(len(clip), dtype=np.int64) - 1
    for k in range(3):
        c = clip[:, k]
        code = (c[:, 0] > c[:, 3]) * 1 + (c[:, 0] < -c[:, 3]) * 2 + (c[:, 1] > c[:, 3]) * 4 + (c[:, 1] < -c[:, 3]) * 8
        side &= code
    keep = side == 0
    pieces = [clip[keep & ~needs]]
    for t in np.nonzero(keep & needs)[0]:
        pieces += [p[None] for p in clip_near_far(clip[t])]
    tri = np.concatenate(pieces) if len(pieces) > 1 else pieces[0]
    hw, hh = w * 0.5, h * 0.5
    r = 1.0 / tri[:, :, 3]
    sx = np.floor((tri[:, :, 0] * r * hw + hw) * 256.0 + 0.5).astype(np.int64)
    sy = np.floor((tri[:, :, 1] * r * hh + hh) * 256.0 + 0.5).astype(np.int64)
    area2 = (sx[:, 1] - sx[:, 0]) * (sy[:, 2] - sy[:, 0]) - (sy[:, 1] - sy[:, 0]) * (sx[:, 2] - sx[:, 0])
    px0 = np.maximum(0, (sx.min(1) - 128 + 255) >> 8); px1 = np.minimum(w - 1, (sx.max(1) - 128) >> 8)
    py0 = np.maximum(0, (sy.min(1) - 128 + 255) >> 8); py1 = np.minimum(h - 1, (sy.max(1) - 128) >> 8)
    vis = (area2 < 0) & (px0 <= px1) & (py0 <= py1)
    sx, sy = sx[vis], sy[vis]
    A = np.zeros((len(sx), 3), np.int64); B = np.zeros_like(A); C = np.zeros_like(A)
    for e in range(3):
        ia, ib = (e + 1) % 3, (e + 2) % 3
        dx, dy = sx[:, ib] - sx[:, ia], sy[:, ib] - sy[:, ia]
        tl = ((dy == 0) & (dx < 0)) | (dy > 0)
        A[:, e], B[:, e], C[:, e] = dy, -dx, dx * sy[:, ia] - dy * sx[:, ia] - np.where(tl, 0, 1)
    return A, B, C, px0[vis], px1[vis], py0[vis], py1[vis]


def count_view(A, B, C, x0, x1, y0, y1):
    ntx = (x1 >> 5) - (x0 >> 5) + 1
    nty = (y1 >> 2) - (y0 >> 2) + 1
    n = ntx * nty
    t = np.repeat(np.arange(len(n)), n)
    r = np.arange(n.sum()) - np.repeat(np.cumsum(n) - n, n)
    tx = (x0 >> 5)[t] + r % ntx[t]
    ty = (y0 >> 2)[t] + r // ntx[t]
    bx0, bx1 = np.maximum(x0[t], tx * 32), np.minimum(x1[t], tx * 32 + 31)
    by0, by1 = np.maximum(y0[t], ty * 4), np.minimum(y1[t], ty * 4 + 3)
    kept = np.ones(len(t), bool)
    for e in range(3):
        a, b = A[t, e], B[t, e]
        f = C[t, e] + a * (np.where(a > 0, bx1, bx0) * 256 + 128) + b * (np.where(b > 0, by1, by0) * 256 + 128)
        kept &= f >= 0
    # exact coverage of the tile's 128 samples, pair by pair
    xs = (np.arange(32) * 256 + 128)[None, None, :]
    ys = (np.arange(4) * 256 + 128)[None, :, None]
    cov = np.ones((len(t), 4, 32), bool)
    for e in range(3):
        f = C[t, e][:, None, None] + A[t, e][:, None, None] * (xs + (tx * 32 * 256)[:, None, None]) + B[t, e][:, None, None] * (ys + (ty * 4 * 256)[:, None, None])
        cov &= f >= 0
    ncov = cov.reshape(len(t), -1).sum(1)
    return len(A), len(t), int(kept.sum()), int((ncov > 0).sum()), int(((ncov > 0) & (ncov <= 4)).sum()), int((~kept & (ncov > 0)).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenario", default="Collect")
    ap.add_argument("--envs", type=int, default=1024)
    ap.add_argument("--agents", type=int, default=4)
    ap.add_argument("--steps", type=int, default=0, help="random steps after the reset")
    ap.add_argument("--views", type=int, default=0, help="count only every k-th view to reach about this many (0: all)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--w", type=int, default=128)
    ap.add_argument("--h", type=int, default=72)
    a = ap.parse_args()
    o = orc.Oracle(a.scenario, a.envs, a.agents, a.w, a.h, render=False)
    o.seed(a.seed)
    o.reset()
    rng = np.random.default_rng(a.seed)
    for _ in range(a.steps):
        o.step(rng.integers(0, 1 << 10, size=a.envs * a.agents, dtype=np.int32) & (1 << rng.integers(0, 10, size=a.envs * a.agents)))
    proj = projection(a.w, a.h)
    N = a.envs * a.agents
    stride = max(1, N // a.views) if a.views else 1
    rows = []
    for v in range(0, N, stride):
        e, ag = divmod(v, a.agents)
        A, B, C, x0, x1, y0, y1 = setup(view_triangles(o.view(e, ag), o.instances(e), a.w, a.h, proj), a.w, a.h)
        rows.append(count_view(A, B, C, x0, x1, y0, y1))
    o.close()
    r = np.array(rows, dtype=np.float64)
    names = ["list", "box", "kept", "covered", "small", "dropped_covered"]
    print("%s %dx%d, %d of %d views, %dx%d: per view mean (min / max)" % (a.scenario, a.envs, a.agents, len(rows), N, a.w, a.h))
    for i, nme in enumerate(names):
        print("  %-16s %9.1f  (%d / %d)" % (nme, r[:, i].mean(), r[:, i].min(), r[:, i].max()))
    box = r[:, 1].sum()
    print("  of the box pairs: kept %.1f %%, covered %.1f %%, small %.1f %%" % (100 * r[:, 2].sum() / box, 100 * r[:, 3].sum() / box, 100 * r[:, 4].sum() / box))
    assert r[:, 5].sum() == 0, "the bin test dropped a covered pair"


if __name__ == "__main__":
    main()
