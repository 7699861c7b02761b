"""The resolve of supersampled images (oracle/ssaa_oracle.py; CRB_SS2 / CRB_SS4, DESIGN 2) on the CPU: the NumPy statement
against a scalar restatement of the rule on random and adversarial blocks, s = 1, constant frames, and a block half covered
by a textured triangle drawn with the pinned oracle."""
import math

import numpy as np
import pytest

F32 = np.float32


def SS():
    from oracle import ssaa_oracle
    return ssaa_oracle


def _tree(vals):
    """((a+b)+(c+d)) of float32 scalars, each addition rounded to float32"""
    vals = [F32(x) for x in vals]
    while len(vals) > 1:
        vals = [F32(vals[i] + vals[i + 1]) for i in range(0, len(vals), 2)]
    return vals[0]


def _to_u8(x):
    """run.py's .astype('uint8') on x86-64: truncate toward zero through int32 (NaN and values outside int range: INT_MIN),
    then the low byte"""
    x = float(x)
    if math.isnan(x) or not (-2147483648.0 <= x < 2147483648.0):
        return 0
    return int(x) & 255


def scalar_resolve(colour, s):
    """The rule, one output element at a time: row sums over the block's columns, then the tree over the row sums"""
    colour = np.asarray(colour, F32)
    H, W = colour.shape[0] // s, colour.shape[1] // s
    means = np.zeros((H, W, 3), F32)
    img = np.zeros((H, W, 3), np.uint8)
    with np.errstate(invalid="ignore", over="ignore"):
        for r in range(H):
            for x in range(W):
                for k in range(3):
                    rows = [_tree(colour[s * r + i, s * x:s * x + s, k]) for i in range(s)]
                    m = F32(_tree(rows) * F32(1.0 / (s * s)))
                    means[r, x, k] = m
                    img[H - 1 - r, x, k] = _to_u8(m)
    return means, img


def _adversarial(seed, H, W):
    rng = np.random.default_rng(seed)
    c = (rng.random((H, W, 3), dtype=F32) * F32(300) - F32(20)).astype(F32)
    specials = np.array([np.nan, np.inf, -np.inf, -0.0, 0.0, 2.0 ** 31, 3e9, -3e9, 2.0 ** 32 + 7, 255.99998, 256.0, -1.5,
                         1e38, 3.4e38, -3.4e38, 2.0 ** 25, 2.0, 1e-45], F32)
    mask = rng.random((H, W, 3)) < 0.3
    c[mask] = rng.choice(specials, size=int(mask.sum()))
    return c


@pytest.mark.parametrize("s", [2, 4])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_numpy_resolve_equals_scalar_rule(seed, s):
    c = _adversarial(seed, 8 * s, 12 * s)
    means, img = scalar_resolve(c, s)
    got = SS().block_means(c, s)
    nan = np.isnan(means)              # (which NaN an operation returns is the hardware's choice; every NaN gives 0)
    assert np.array_equal(np.isnan(got), nan) and nan.any()
    assert np.array_equal(got[~nan].view(np.uint32), means[~nan].view(np.uint32))
    assert np.array_equal(SS().resolve(c, s), img)


def test_tree_order_is_not_left_to_right():
    """Blocks whose pairwise tree and left-to-right sums round differently: the resolve follows the tree."""
    for s, block in ((2, [[2.0 ** 25, 2.0], [2.0, 2.0]]),
                     (4, [[2.0 ** 25, 2.0, 2.0, 2.0], [2.0, 2.0, 2.0, 2.0], [2.0, 2.0, 2.0, 2.0], [2.0, 2.0, 2.0, 2.0]])):
        b = np.asarray(block, F32)
        c = np.repeat(b[:, :, None], 3, axis=2)
        left = F32(0)
        for x in b.ravel():
            left = F32(left + x)
        tree = _tree([_tree(row) for row in b])
        assert tree != left
        want = _to_u8(F32(tree * F32(1.0 / (s * s))))
        assert want != _to_u8(F32(left * F32(1.0 / (s * s))))
        assert (SS().resolve(c, s) == want).all()
        assert np.array_equal(SS().resolve(c, s), scalar_resolve(c, s)[1])


def test_nan_and_inf_propagate():
    c = np.zeros((2, 4, 3), F32)
    c[0, 0] = [np.nan, np.inf, np.inf]
    c[1, 1, 2] = -np.inf                  # inf + -inf = NaN
    c[0, 2] = [np.inf, -0.0, -0.0]
    m = SS().block_means(c, 2)
    assert np.isnan(m[0, 0, 0]) and m[0, 0, 1] == np.inf and np.isnan(m[0, 0, 2])
    assert m[0, 1, 0] == np.inf and np.signbit(m[0, 1, 1]) is np.False_    # -0 + -0 + +0 + +0 = +0
    assert (SS().resolve(c, 2)[0, :1] == 0).all()


def test_s1_is_the_flipped_truncation():
    c = _adversarial(5, 24, 40)
    with np.errstate(invalid="ignore"):
        assert np.array_equal(SS().resolve(c, 1), c[::-1].astype("uint8"))


@pytest.mark.parametrize("s", [2, 4])
def test_constant_frame_resolves_to_itself(s):
    rng = np.random.default_rng(s)
    for k in range(4):
        val = (rng.random(3, dtype=F32) * F32(600) - F32(100)).astype(F32)
        one = np.broadcast_to(val, (6, 10, 3)).astype(F32)
        with np.errstate(invalid="ignore"):
            assert np.array_equal(SS().resolve(np.broadcast_to(val, (6 * s, 10 * s, 3)), s), one[::-1].astype("uint8"))


@pytest.mark.parametrize("s", [2, 4])
def test_half_covered_block_resolves_to_the_mean(s):
    """A quad with a constant 1 x 1 texture (every covered sample is exactly the texel) whose right edge falls inside a block
    column: blocks with k of s*s samples covered resolve to trunc(texel * k / s^2); the half-covered column is there."""
    h = w = 8
    S = s * w
    edge = S // 2 + s // 2 - 0.5          # screen x of the edge: samples up to S/2 + s/2 - 1 covered, half of block column w/2
    x_edge = F32(2) * (F32(edge) / F32(S // 2) - F32(1))      # screen x = (x/z + 1) * S/2 at z = 2
    z = F32(2)
    v = np.array([[[-50, -50, z], [x_edge, -50, z], [-50, 50, z]], [[x_edge, -50, z], [x_edge, 50, z], [-50, 50, z]]], F32)
    n = np.zeros_like(v)
    n[..., 2] = -1
    uv = np.full_like(v, 0.5)
    tex = np.array([[[200, 100, 50]]], np.uint8)
    o = SS().sample_frame(h, w, s, v, uv, n, texture=tex)
    covered = o.z_buffer < F32(1e6)
    assert covered.any() and not covered.all()
    assert np.array_equal(np.unique(o.color_buffer[covered], axis=0), [[200.0, 100.0, 50.0]])
    img = SS().resolve(o.color_buffer, s)
    k = covered.reshape(h, s, w, s).sum(axis=(1, 3))
    assert (k == s * s // 2).any(), "no half-covered block"
    want = (np.array([200, 100, 50])[None, None, :] * k[:, :, None] // (s * s)).astype(np.uint8)[::-1]
    assert np.array_equal(img, want)
    assert np.array_equal(SS().render_resolved(h, w, s, v, uv, n, texture=tex), img)


def test_refuses_other_factors():
    for s in (0, 3, 8):
        with pytest.raises(ValueError):
            SS().block_means(np.zeros((8, 8, 3), F32), s)
    with pytest.raises(ValueError):
        SS().block_means(np.zeros((6, 8, 3), F32), 4)
