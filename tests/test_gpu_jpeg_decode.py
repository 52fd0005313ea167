"""JPEG reader (SURVEY.md 8f-2) on the GPU through the C-ABI: rt_jpeg_decode (host Huffman + device IDCT / up-sampling /
colour conversion) must return the float image stbi_loadf returns (main.cu:376-380) — byte / 255.f of stb's decode, bit
for bit: against the committed stb outputs, the CPU oracle, and the earth texture as a JPEG file."""
import numpy as np
import pytest

import raytracing_renderer_cuda_b200 as rt
from raytracing_renderer_cuda_b200 import capi
from tests import oracle_api as oa
from tests.conftest import ROOT

pytestmark = pytest.mark.gpu
EARTH_JPG = ROOT / "oracle" / "_ref" / "textures" / "earth.jpg"  # the reference's own texture, where `make -C oracle ref` ran


@pytest.fixture(scope="module")
def ctx():
    return rt.Context(0)


def _as_float(pix: np.ndarray) -> np.ndarray:
    return pix.astype(np.float32) / np.float32(255.0)  # stbi__ldr_to_hdr with gamma = scale = 1


@pytest.fixture(scope="module")
def earth_jpg(earth, tmp_path_factory):
    """The C1 earth texture as a file of the kind the reference's main() opens (textures/earth.jpg: progressive, 4:2:0,
    1200x600), encoded from the committed asset -> (path, the bytes the CPU reader decodes from it, pinned to stb by
    tests/test_jpeg_decode.py)."""
    import io
    from PIL import Image

    b = io.BytesIO()
    Image.fromarray(np.round(earth * 255.0).astype(np.uint8)).save(b, "JPEG", quality=90, progressive=True, subsampling=2)
    path = tmp_path_factory.mktemp("textures") / "earth.jpg"
    path.write_bytes(b.getvalue())
    c = capi.jpeg_parse(b.getvalue())
    try:
        assert c.contents.progressive == 1 and (c.contents.h_max, c.contents.v_max) == (2, 2)
        pix = oa.oracle_jpeg_pixels(c)
    finally:
        capi.jpeg_coefficients_free(c)
    return path, pix


def test_device_reader_equals_stb_fixtures(ctx):
    g = np.load(ROOT / "tests" / "golden" / "jpeg_decode_golden.npz")
    n = 0
    for key in sorted(k for k in g.files if k.startswith("file")):
        got, ms = capi.jpeg_decode(ctx, g[key].tobytes())
        want = _as_float(g[f"pix{key[4:]}"])
        assert got.shape == want.shape and np.array_equal(got, want), str(g[f"name{key[4:]}"])
        n += 1
    assert n >= 50


def test_device_pixel_stages_equal_the_oracle_on_larger_frames(ctx):
    import io
    from PIL import Image

    for (w, h, prog, sub) in [(1201, 599, True, 2), (640, 360, False, 1), (777, 333, True, 0), (1920, 1080, False, 2)]:
        img = oa.jpeg_test_image("photo", w, h, seed=w)
        b = io.BytesIO()
        Image.fromarray(img).save(b, "JPEG", quality=90, progressive=prog, subsampling=sub)
        c = capi.jpeg_parse(b.getvalue())
        want = _as_float(oa.oracle_jpeg_pixels(c))
        capi.jpeg_coefficients_free(c)
        got, ms = capi.jpeg_decode(ctx, b.getvalue())
        assert np.array_equal(got, want) and ms > 0, (w, h, prog, sub)


def test_reference_texture_is_ingested_bit_exact(ctx, earth, earth_jpg):
    """The earth texture as a progressive 4:2:0 JPEG file through the device reader and through rt_image_load (the path
    a scene file or the app takes) == byte / 255.f of what the stb-pinned CPU reader decodes from the same file.  Where
    the reference has been built (oracle/_ref/), also its own textures/earth.jpg == the stb-decoded asset the scenes use,
    so a scene built from that JPEG file is the scene built from assets/earth_stb.png."""
    import ctypes as C

    cases = [(earth_jpg[0], _as_float(earth_jpg[1]))]
    if EARTH_JPG.exists():
        cases.append((EARTH_JPG, earth))
    for path, want in cases:
        got, _ = capi.jpeg_decode(ctx, path.read_bytes())
        assert got.shape == (600, 1200, 3)
        assert np.array_equal(got, want), path
        px, w, h = C.POINTER(C.c_float)(), C.c_int32(), C.c_int32()
        assert ctx.lib.rt_image_load(ctx._h, str(path).encode(), C.byref(px), C.byref(w), C.byref(h)) == capi.RT_OK
        loaded = np.ctypeslib.as_array(px, (h.value, w.value, 3)).copy()
        ctx.lib.rt_free(px)
        assert np.array_equal(loaded, want), path


def test_round_trip_with_the_device_writer(ctx):
    """device JPEG writer -> device JPEG reader: the quality-100 file of a frame decodes to within the quantiser's error."""
    img = oa.jpeg_test_image("photo", 320, 200, seed=9)
    back, _ = capi.jpeg_decode(ctx, capi.jpeg_encode(ctx, img, 100))
    assert back.shape == (200, 320, 3)
    assert np.abs(back * 255.0 - img.astype(np.float32)).max() <= 6.0


def test_cpp_app_reads_the_jpeg_texture_like_the_reference_main(tmp_path, earth_jpg):
    """apps/render_scene with --earth earth.jpg (a file like the one the reference's main() opens, main.cu:134,380)
    renders the same frame as with a PPM of the bytes decoded from it: one sample per pixel, so the two frames are
    bit-identical."""
    import subprocess

    path, pix = earth_jpg
    ppm = tmp_path / "earth.ppm"
    ppm.write_bytes(b"P6\n%d %d\n255\n" % (pix.shape[1], pix.shape[0]) + pix.tobytes())
    app = ROOT / "apps" / "render_scene"
    outs = []
    for earth_arg in (str(path), str(ppm)):
        out = tmp_path / f"f{len(outs)}.ppm"
        r = subprocess.run([str(app), "--scene", "earth_emitter", "--width", "300", "--height", "150", "--spp", "1", "--out", str(out),
                            "--earth", earth_arg], capture_output=True, text=True, cwd=str(ROOT))
        assert r.returncode == 0, r.stdout + r.stderr
        outs.append(out.read_bytes())
    assert outs[0] == outs[1]


def test_json_scene_with_a_jpeg_texture(ctx, earth_jpg):
    """A scene document may name a JPEG file once the front-end has a context: C1 with earth.jpg flattens to the same
    description as the hard-coded scene with the image decoded from that file."""
    import ctypes as C
    import json

    path, pix = earth_jpg
    doc = json.loads((ROOT / "assets" / "scenes" / "earth_emitter.json").read_text())
    doc["textures"]["earth"]["file"] = str(path)
    d = rt.SceneDesc.from_json(json.dumps(doc), ctx=ctx)
    b = rt.SceneDesc.builtin("earth_emitter", _as_float(pix))
    ia, ib = d.desc.images[0], b.desc.images[0]
    assert (ia.width, ia.height) == (ib.width, ib.height) == (1200, 600)
    n = 1200 * 600 * 3
    assert np.array_equal(np.ctypeslib.as_array(ia.rgb, (n,)), np.ctypeslib.as_array(ib.rgb, (n,)))
    with pytest.raises(capi.RtError):
        rt.SceneDesc.from_json(json.dumps(doc))  # without a context a JPEG cannot be read
