"""GPU drop-in proof (-m gpu): the reference's OWN types and draw-call signatures (DTRRenderContext,
DTRRenderTransform, DTRMesh, DqnV*) drive the CUDA back end through the host-side mirror
dtrenderer_b200/host/DTRRenderB200.h, inside the same headless harness that drives the unmodified
reference.  oracle/_ref/libdtr_ref_b200.so must produce the reference's frames and work counters: those
stored in tests/golden/digests.json (outputs of the unmodified reference), and, where the reference itself
is built (oracle/_ref/libdtr_ref.so), its live frames as well.  Without the reference sources the harness is
built against the stand-in declarations of its types in oracle/ref_types/."""
import numpy as np
import pytest

from dtrenderer_b200 import scenes
from golden_scenes import DIGESTS, SCENES, digest

pytestmark = pytest.mark.gpu

NAMES = ["cfg1_800x600", "edges_320x200", "lines_256x192", "text_320x200", "odd_333x217", "flat_640x480",
         "cfg3_textured_overlays_720p", "view_37_of_4096_640x360"]


def _harness():
    from oracle import dtro
    assert dtro.available("reference_api_b200"), "oracle/_ref/libdtr_ref_b200.so not built (make -C oracle ref)"
    return dtro


@pytest.mark.parametrize("name", NAMES)
def test_reference_api_on_b200_matches_reference(built, name):
    dtro = _harness()
    w, h, make = SCENES[name]
    scene = make()
    gpu = dtro.Oracle(w, h, "reference_api_b200")
    assert gpu.lib.dtro_kind() == b"reference-api-on-b200"
    gpu.reset_counters()
    scenes.replay(scene, gpu)
    if dtro.available("reference"):
        ref = dtro.Oracle(w, h, "reference")
        ref.reset_counters()
        scenes.replay(scene, ref)
        assert np.array_equal(gpu.zbuffer().view(np.uint32), ref.zbuffer().view(np.uint32))
        assert np.array_equal(gpu.color(), ref.color())
        assert gpu.counters() == ref.counters()
    g = DIGESTS[name]
    assert digest(gpu.zbuffer()) == g["depth_sha256"], "depth plane differs from the reference's"
    assert digest(gpu.color()) == g["color_sha256"], "colour plane differs from the reference's"
    assert gpu.counters() == (g["setPixels"], g["triangles"])


def test_two_frames_keep_colour_and_reset_depth(built):
    """Frame protocol of DTR_Update: depth is reset every frame, colour persists until cleared."""
    dtro = _harness()
    w, h = 320, 200
    outs = []
    # the unmodified reference where it is built, else the C restatement pinned to it (tests/test_oracle_pinning.py)
    for kind in ("reference" if dtro.available("reference") else "port", "reference_api_b200"):
        o = dtro.Oracle(w, h, kind)
        scenes.replay(scenes.cfg1_scene(w, h), o)
        o.color()  # present frame 1
        o.reset_z()  # frame 2: no clear, draws on top of frame 1's colour
        o.triangle(np.asarray((20, 20, 3, 300, 40, 3, 150, 190, 3), np.float32), (0.2, 0.4, 0.9, 0.6))
        outs.append((o.color().copy(), o.zbuffer().copy()))
    assert np.array_equal(outs[0][0], outs[1][0])
    assert np.array_equal(outs[0][1].view(np.uint32), outs[1][1].view(np.uint32))
