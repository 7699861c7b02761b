"""The id-output oracle (oracle/ids_oracle.py) against oracle_render's own buffers, on the CPU.

The oracle composes winner_ids and _bary (texture_mip_oracle).  Restating z, normals and per-vertex colour from its
(tri_id, bary) with the projected / per-corner arrays, with left-associated sums, must give oracle_render's buffers bit for
bit at every pixel a call wrote, and -1 must appear exactly where no call wrote.  "Wrote" is read off a colour buffer
pre-filled with a NaN sentinel: the z-test does not look at colour, so the sentinel survives exactly where nothing was drawn.
"""
import numpy as np
import pytest

from conftest import TriModel, bits_equal, load_indexed, random_scene

F32 = np.float32
SENTINEL = np.uint32(0x7FC0DEAD)


def _ids():
    from oracle import ids_oracle
    return ids_oracle


def _O():
    from oracle import oracle
    return oracle


def _filler(h, w, fov):
    o = _ids().IdsOracleFiller(h, w, fov=fov)
    o.color_buffer.view(np.uint32)[:] = SENTINEL
    return o


def _written(o):
    return (o.color_buffer.view(np.uint32) != SENTINEL).any(axis=2)


def _check_call(o, m, base, where):
    """z, normals and colour of the pixels this call's ids claim, restated from (tri_id, bary), equal the buffers."""
    I, O = _ids(), _O()
    v, c, n = m._vertices_by_triangles, m._colors_by_triangles, m._normals_by_triangles
    scr = O.project(o.h, o.w, o.proj_mat.ravel(), v)
    sel = (o.tri_id >= base) & (o.tri_id < base + len(v)) & where
    z = I.restate(scr[..., 2:3], o.tri_id, o.bary, base)[..., 0]
    nb = I.restate(n, o.tri_id, o.bary, base)
    cb = I.restate(c, o.tri_id, o.bary, base)
    assert bits_equal(z[sel], o.z_buffer[sel])
    assert bits_equal(nb[sel], o.normals_buffer[sel])
    assert bits_equal(cb[sel], o.color_buffer[sel])
    return int(sel.sum())


def _single(m, h, w, fov):
    o = _filler(h, w, fov)
    o.render_model(m)
    wr = _written(o)
    assert np.array_equal(o.tri_id == -1, ~wr)
    assert (o.tri_id < len(m._vertices_by_triangles)).all()
    assert bits_equal(o.bary[~wr], np.zeros((int((~wr).sum()), 3), F32))
    return _check_call(o, m, 0, wr)


@pytest.mark.parametrize("name,size,fov", [("trex", 256, 45.0), ("bunny", 200, 60.0), ("basketball", 160, 90.0)])
def test_restated_buffers_on_golden_fixtures(name, size, fov):
    assert _single(load_indexed(name), size, size, fov) > 500


@pytest.mark.parametrize("seed", range(10))
def test_restated_buffers_on_random_scenes(seed):
    _single(random_scene(seed), 96, 128, 90.0)


def test_two_composited_calls_with_different_bases():
    a, b = random_scene(3, T=300), random_scene(4, T=250)
    o = _filler(96, 128, 90.0)
    o.render_model(a, base=0)
    o.render_model(b, base=1000)
    wr = _written(o)
    assert np.array_equal(o.tri_id == -1, ~wr)
    ida = (o.tri_id >= 0) & (o.tri_id < 300)
    idb = (o.tri_id >= 1000) & (o.tri_id < 1250)
    assert np.array_equal(ida | idb, wr)
    assert _check_call(o, a, 0, wr) > 0 and _check_call(o, b, 1000, wr) > 0


def _quad_pair(z, colours):
    """Two copies of the same screen-filling triangle pair at depth z (camera space), one colour per copy."""
    v = np.array([[[-1, -1, z], [1, -1, z], [-1, 1, z]], [[1, -1, z], [1, 1, z], [-1, 1, z]]], F32)
    v = np.concatenate([v, v])
    n = np.zeros_like(v)
    n[..., 2] = -1
    c = np.concatenate([np.full((2, 3, 3), col, F32) for col in colours])
    return TriModel(v, c, n)


def test_equal_depth_ties():
    m = _quad_pair(2.0, (10.0, 20.0))
    o = _filler(32, 32, 90.0)
    o.render_model(m)
    wr = _written(o)
    assert wr.sum() >= 200
    assert set(np.unique(o.tri_id[wr])) <= {2, 3}            # within a call the highest index wins
    assert (o.color_buffer[wr] == 20.0).all()
    o.render_model(_quad_pair(2.0, (30.0, 40.0)), base=100)
    assert set(np.unique(o.tri_id[wr])) <= {102, 103}        # across calls the later call wins
    assert (o.color_buffer[wr] == 40.0).all()
    o.render_model(_quad_pair(3.0, (50.0, 60.0)), base=200)   # behind: nothing is written, the ids stay
    assert set(np.unique(o.tri_id[wr])) <= {102, 103}
    assert np.array_equal(o.tri_id == -1, ~wr)
