"""The raster kernel bins each batch of triangles to its 32x4-pixel tiles before it draws them, with a conservative integer test of every
edge against the tile (a pair is dropped only when one edge function is negative at every sample of the tile).  These scenes put that
test where it can go wrong: triangle edges and vertices exactly on tile borders (pixel x a multiple of 32, pixel y a multiple of 4),
edges through the sample centres of a tile's first and last column or row (the top-left rule decides those samples), thin slivers
whose pixel boxes span many tiles they never touch, and the largest band (128 tiles) with the longest triangle list (1022), where the
bins of a band take more than one round.  Every frame is compared with the oracle byte for byte."""
import numpy as np
import pytest

import helpers

W, H = 128, 72
F32 = np.float32


def _projection(w, h):
    aspect = F32(w) / F32(h)
    half_tan = F32(np.tan(np.float64(F32(100.0) * F32(0.01745329251994329576923690768489)) / 2.0))
    return F32(1.0) / half_tan, -aspect / half_tan


def _facing_box(k, px0, py0, px1, py1, z_front, half_z):
    """a box facing the camera (identity view) whose front face spans window x px0..px1, y py0..py1 (in pixels, fractional allowed)"""
    p00, p11 = _projection(W, H)
    x0, x1 = [(px - W / 2) / (W / 2) * (-z_front) / float(p00) for px in (px0, px1)]
    y0, y1 = [(py - H / 2) / (H / 2) * (-z_front) / float(p11) for py in (py0, py1)]
    m = np.eye(4)
    m[0, 0], m[1, 1], m[2, 2] = abs(x1 - x0) / 2, abs(y1 - y0) / 2, half_z
    m[:3, 3] = [(x0 + x1) / 2, (y0 + y1) / 2, z_front - half_z]
    return np.concatenate([[0, k % 20], m.T.reshape(-1)])


def _render_both(view16, inst):
    import orc
    from megaverse_b200 import capi

    rgba_o, depth_o = orc.render_instances(view16, inst, W, H, want_depth=True)
    rgba_g, depth_g = capi.render_instances(view16, inst, W, H, want_depth=True)
    return rgba_o, depth_o, np.asarray(rgba_g), np.asarray(depth_g)


def _assert_same(view16, inst, min_covered):
    rgba_o, depth_o, rgba_g, depth_g = _render_both(view16, inst)
    assert (depth_o > 0).sum() >= min_covered, "the scene should cover pixels"
    bad = (rgba_o != rgba_g).any(axis=-1)
    assert not bad.any(), "colour differs in %d pixels, first at %s" % (int(bad.sum()), np.argwhere(bad)[:4].tolist())
    assert np.array_equal(depth_o.view(np.uint32), depth_g.view(np.uint32)), "depth differs in %d pixels" % int((depth_o != depth_g).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 0.5])
def test_edges_and_vertices_on_tile_borders(built, offset):
    """offset 0: box corners on tile corners (edges along the borders between tiles, no sample on them); offset 0.5: edges through the
    sample centres of the first or last column / row of a tile -- ties the top-left rule decides -- and vertices on those centres"""
    rows = []
    spans = [(32, 4, 64, 8), (31, 3, 64, 12), (0, 0, 32, 4), (64, 8, 96, 36), (95, 35, 128, 72), (32, 40, 33, 44), (96, 4, 97, 68)]
    for k, (x0, y0, x1, y1) in enumerate(spans):
        rows.append(_facing_box(k, x0 + offset, y0 + offset, x1 + offset, y1 + offset, -3.0 - 0.7 * k, 0.3))
    # the two triangles of a square face share a diagonal from tile corner to tile corner
    rows.append(_facing_box(9, 32 + offset, 8 + offset, 64 + offset, 40 + offset, -2.0, 0.2))
    view16 = np.eye(4, dtype=F32).reshape(-1)
    _assert_same(view16, np.array(rows, dtype=F32), 500)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_slivers_spanning_many_tiles(built, seed):
    """long thin rods at steep angles: their triangles' pixel boxes cover many tiles, the triangles only a few of them"""
    rng = np.random.default_rng(4000 + seed)
    rows = []
    for k in range(12):
        m = np.eye(4)
        ang = rng.uniform(0, np.pi)
        c, s = np.cos(ang), np.sin(ang)
        tilt = rng.uniform(-0.6, 0.6)
        rot = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]]) @ np.array([[1, 0, 0], [0, np.cos(tilt), -np.sin(tilt)], [0, np.sin(tilt), np.cos(tilt)]])
        m[:3, :3] = rot @ np.diag([rng.uniform(2.0, 6.0), rng.uniform(0.005, 0.03), rng.uniform(0.005, 0.03)])
        m[:3, 3] = [rng.uniform(-2, 2), rng.uniform(-1, 1), -rng.uniform(4.0, 8.0)]
        rows.append(np.concatenate([[0, k], m.T.reshape(-1)]))
    rows.append(_facing_box(19, 10, 6, 118, 66, -12.0, 0.5))  # a backdrop, so that the slivers also win and lose depth tests
    view16 = np.eye(4, dtype=F32).reshape(-1)
    _assert_same(view16, np.array(rows, dtype=F32), 2000)


@pytest.mark.gpu
def test_largest_band_and_longest_list(built):
    """128 tiles in one band (256 x 64, one band per view) with a triangle list of 1022 entries: shared memory then holds the bins of
    fewer tiles than the band has, and the band is binned and drawn in rounds.  Frames equal the oracle's; the binning's pair counters
    say that it evaluated no more (tile, triangle) pairs than the pixel boxes hold."""
    import orc
    from megaverse_b200 import capi

    E, A, w, h = 4, 2, 256, 64
    o = orc.Oracle("Collect", E, A, w, h)
    g = capi.Engine("Collect", E, A, w, h, num_threads=2)
    g.set_option("fast_shading", 0)
    g.set_option("tri_cap", 1022)
    g.set_option("raster_bands", 1)
    o.seed(5); g.seed(5); o.reset(); g.reset()
    g.raster_stats(enable=True, read=False)
    rng = np.random.default_rng(3)
    for t in range(12):
        acts = helpers.purposeful_actions(rng, E * A, t)
        o.step(acts); g.step(acts)
        a, b = o.obs(), np.array(g.obs())
        assert np.array_equal(a, b), "step %d: %d pixels differ" % (t, int((a != b).any(axis=-1).sum()))
    st = g.raster_stats(enable=False, read=True)
    assert st["work_items"] > 0 and st["pairs_in_boxes"] > 0, "the counters were on"
    assert 0 < st["pairs_evaluated"] <= st["pairs_in_boxes"], st
    assert g.faults() == 0
    o.close(); g.close()
