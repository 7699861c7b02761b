"""seeded_checksums.json: what the reference computed on the seeded inputs of the tests that compare with its own code.

Those tests (tests/test_oracle_pinning.py, test_ingest_oracle.py, test_gpu_parity.py) compare with the reference's own
classes where oracle/_ref is present (oracle/build_ref.py builds it from a checkout of the reference).  The checksums here
let them compare with the reference's results everywhere else.  They are computed by the oracle, which the project pinned
bit-equal to the reference build on exactly these inputs (DESIGN.md section 1, row (c), and section 4b):
  * random_scenes / out_of_range: OracleFiller on the 24 seeded random scenes and on the out-of-range-coordinate scene;
  * random_meshes: the ingest oracle's vertex normals, vertex colours and gathers of the 6 seeded random meshes (sha256 with
    every NaN written as 0x7FC00000: NaN bits are not part of the contract);
  * renderer_flow_*: run.py's Renderer.render flow (render_model, Guro illumination in place, colour buffer) on the oracle;
    its Guro step is pinned to the reference's lit-colour goldens in checksums.json.
Run from the repository root after build(): python tests/golden/make_golden_seeded.py
"""
import json
import os
import sys
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, TESTS)
sys.path.insert(0, os.path.dirname(TESTS))

from conftest import load_indexed  # noqa: E402
from oracle import ingest as I  # noqa: E402
from oracle import oracle as O  # noqa: E402
import test_gpu_parity as GP  # noqa: E402
import test_ingest_oracle as IO  # noqa: E402
import test_oracle_pinning as OP  # noqa: E402


def random_scenes():
    out = {}
    for seed in range(24):
        h, w, fov, m, passes = OP.random_scene_case(seed)
        f = O.OracleFiller(h, w, fov=fov)
        for _ in range(passes):
            f.render_model(m)
        out[str(seed)] = OP.buffer_sums(f)
    return out


def out_of_range():
    f = O.OracleFiller(64, 64, fov=90.0)
    f.render_model(OP.out_of_range_model())
    return {"z": OP.sha(f.get_z_buffer()), "color": OP.sha(f.get_color_buffer())}


def random_meshes():
    out = {}
    for seed in range(6):
        v, tri, vt, tvt, tex, invert = IO.random_mesh(seed)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            n = I.vertex_normals(v, tri, invert=invert)
        c = I.vertex_colors(vt, tex)
        out[str(seed)] = IO.mesh_sums(n, c, I.gather(n, tri), I.gather(c, tvt))
    return out


def renderer_flow(models, h, w, light):
    """Renderer.render (renderer.py:47-49) once per model on one filler; light None = NoIllumination."""
    f = O.OracleFiller(h, w, fov=45)
    frames = []
    for m in models:
        f.render_model(m)
        if light is not None:
            O.guro(f.get_color_buffer(), f.get_normals_buffer(), light)
        frames.append(GP.flow_sums(f.get_color_buffer(), f))
    return frames


def main():
    trex, bunny = load_indexed("trex"), load_indexed("bunny")
    light = [0.3, -0.2, 1.0]
    data = {
        "generator": "tests/golden/make_golden_seeded.py",
        "random_scenes": random_scenes(),
        "out_of_range": out_of_range(),
        "random_meshes": random_meshes(),
        "renderer_flow_trex_256x256_guro": renderer_flow([trex], 256, 256, [0, 0, 1])[0],
        "renderer_flow_trex_bunny_320x256": {"guro": renderer_flow([trex, bunny], 320, 256, light),
                                             "none": renderer_flow([trex, bunny], 320, 256, None)},
    }
    with open(os.path.join(HERE, "seeded_checksums.json"), "w") as fh:
        json.dump(data, fh, indent=1, sort_keys=True)
        fh.write("\n")


if __name__ == "__main__":
    main()
