"""CPU oracle of supersampled images (CRB_SS2 / CRB_SS4, render_views(supersample=s), HostImagePipeline(supersample=s);
DESIGN 2) -- an extension of this project.

TEST INFRASTRUCTURE ONLY.  Composed of pinned pieces, nothing new but the resolve:

  1. oracle_render (OracleFiller.render_arrays) draws the frame at (s*h, s*w) samples -- the filler of that size, and so
     its projection -- or, textured, texture_wrap_oracle.TexturedOracleFiller at that size (every filter, interpolation and
     wrap mode);
  2. oracle.guro lights the colour buffer where the frame is lit;
  3. resolve() states the resolve in NumPy float32: per channel the pairwise tree over each sample row's s columns, then over
     the block's s row sums (`a[..., 0::2, :] + a[..., 1::2, :]`, one binary32 rounding per addition), times F(1/s^2),
     .astype('uint8'), rows flipped.

tests/test_ssaa_oracle.py checks resolve() against a scalar restatement of the rule.
"""
import numpy as np

from oracle import oracle as O
from oracle import texture_wrap_oracle as WR

F32 = np.float32
FACTORS = (1, 2, 4)


def block_means(colour, s):
    """[..., H, W, 3] float32 samples -> [..., H/s, W/s, 3] float32: each s x s block's tree sum times F(1/s^2), rows not
    flipped.  s = 1 returns the samples."""
    if s not in FACTORS:
        raise ValueError(f"s must be 1, 2 or 4, got {s!r}")
    a = np.asarray(colour, F32)
    if a.shape[-3] % s or a.shape[-2] % s:
        raise ValueError(f"{a.shape[-3]} x {a.shape[-2]} samples are not whole {s} x {s} blocks")
    with np.errstate(invalid="ignore", over="ignore"):
        for _ in range(s.bit_length() - 1):            # along each sample row: (a+b), then ((a+b)+(c+d))
            a = a[..., :, 0::2, :] + a[..., :, 1::2, :]
        for _ in range(s.bit_length() - 1):            # then across the block's row sums, the same way
            a = a[..., 0::2, :, :] + a[..., 1::2, :, :]
        return a * F32(1.0 / (s * s))


def resolve(colour, s):
    """The supersampled uint8 image of [..., H, W, 3] float32 samples: [..., H/s, W/s, 3], rows flipped (run.py:26)."""
    m = block_means(colour, s)
    with np.errstate(invalid="ignore"):
        return np.ascontiguousarray(m[..., ::-1, :, :].astype("uint8"))


def sample_frame(h, w, s, v, c, n, fov=90.0, texture=None, filter="nearest", perspective=False, wrap="clamp"):
    """The oracle filler of one fresh frame at (s*h, s*w) samples (output size h x w)."""
    if texture is None:
        o = O.OracleFiller(s * h, s * w, fov=fov)
        o.render_arrays(v, c, n)
    else:
        o = WR.TexturedOracleFiller(s * h, s * w, fov=fov, wrap=wrap)
        o.render_arrays(v, c, n, texture=texture, perspective=perspective, filter=filter)
    return o


def render_resolved(h, w, s, v, c, n, fov=90.0, light=None, **tex):
    """uint8 [h, w, 3]: the supersampled image of one fresh frame of output size h x w, lit with GuroIllumination(light) if
    light is given; `tex` as sample_frame's texture keywords."""
    o = sample_frame(h, w, s, v, c, n, fov=fov, **tex)
    colour = o.color_buffer.copy()
    if light is not None:
        O.guro(colour, o.normals_buffer, light)
    return resolve(colour, s)
