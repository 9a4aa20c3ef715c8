"""CPU: the PNG encoder of dc_png_encode (csrc/png.cu), through its host-compiled test entry point dc_debug_png_host --
every file byte for byte what cv2.imencode(".png", img) writes and what the zlib oracle of tests/png_cases.py builds,
on a corpus that reaches every deflate block type and both code-length limits; the static bounds; argument errors; the
ctypes layout of dc_png_args_t."""
import ctypes as C

import numpy as np
import pytest

import png_cases as pc


def host(img, stats=False):
    from unet_dc_segmentation_b200.png import encode_png_host
    return encode_png_host(img, stats)


def check(img, what=""):
    import cv2
    got, st = host(img, True)
    ok, want = cv2.imencode(".png", img)
    assert ok
    want = want.tobytes()
    assert pc.png_like_cv2(img) == want, f"{what}: the oracle no longer describes this OpenCV"
    assert got == want, f"{what} {img.shape}: {len(got)} bytes, cv2 {len(want)}"
    return st


@pytest.mark.parametrize("shape", pc.SHAPES, ids=[f"{h}x{w}" for h, w in pc.SHAPES])
def test_corpus_equals_opencv(shape):
    for name, img in pc.corpus_for_shape(*shape).items():
        check(img, name)


def test_crafted_streams_and_every_path():
    seen = set()
    stats = {}
    for name, img in pc.crafted().items():
        st = check(img, name)
        stats[name] = st
        seen |= {int(t) & 3 for t in st}
    for name, img in pc.corpus_for_shape(276, 408).items():
        seen |= {int(t) & 3 for t in check(img, name)}
    assert seen == {0, 1, 2}, seen                                    # stored, fixed and dynamic blocks
    assert any(int(t) & 4 for t in stats["fib_15_bits"])              # literal/length lengths limited to 15
    assert any(int(t) & 8 for t in stats["bl_7_bits"])                # bit-length lengths limited to 7
    e = stats["empty_final_block"]
    assert len(e) == 3 and e[-1] & 3 == 1                             # 2 x 16383 symbols, then the empty final block
    for name in ("stored_match_then_dynamic", "uniform_with_line"):   # a stored block with matches, then a coded one
        t = [int(x) & 3 for x in stats[name]]
        assert any(a == 0 and b != 0 for a, b in zip(t, t[1:])), (name, t)


def test_probes_reach_every_block_type():
    from unet_dc_segmentation_b200.png import probe_images
    seen = set()
    for img in probe_images():
        seen |= {int(t) & 3 for t in check(img, "probe")}
    assert seen == {0, 1, 2}, seen


def test_sizes_around_the_window_rewrite():
    # filtered sizes on both sides of libpng's 16384-byte limit and of every halving of the window
    rs = np.random.default_rng(5)
    for n in (127, 128, 129, 255, 256, 257, 1023, 1024, 1025, 8191, 8192, 8193, 16383, 16384, 16385):
        W = n - 1
        check(rs.normal(100, 3, (1, W)).clip(0, 255).astype(np.uint8), f"stream of {n}")
        check(np.zeros((1, W), np.uint8), f"zero stream of {n}")


def test_bounds_hold():
    from unet_dc_segmentation_b200.png import png_bounds
    for shape in pc.SHAPES:
        for name, img in pc.corpus_for_shape(*shape, seed=3).items():
            c = 1 if img.ndim == 2 else 3
            need, ws = png_bounds(1, img.shape[0], img.shape[1], c)
            assert len(host(img)) <= need and ws > 0
    need4, _ = png_bounds(4, 100, 100, 3)
    need1, _ = png_bounds(1, 100, 100, 3)
    assert need4 == 4 * need1
    # a 16k^2 BGR frame: more than 2^32 bits of deflate stream, still in the limits
    need, ws = png_bounds(1, 16384, 16384, 3)
    assert need > 16384 * 16384 * 3 and ws > need


def test_argument_errors():
    from unet_dc_segmentation_b200 import _lib
    from unet_dc_segmentation_b200.png import png_bounds
    for args in [(0, 8, 8, 1), (65536, 8, 8, 1), (1, 0, 8, 1), (1, 8, 0, 1), (1, 8, 8, 2), (1, 8, 8, 4),
                 (1, 32768, 32768, 3)]:
        with pytest.raises(_lib.DcError, match="dc_png_bounds"):
            png_bounds(*args)
    lib = _lib.load()
    out, ws = C.c_int64(), C.c_size_t()
    assert lib.dc_png_bounds(1, 8, 8, 1, None, C.byref(ws)) == _lib.DC_EINVAL
    img = np.zeros((8, 8), np.uint8)
    small = np.empty(16, np.uint8)
    n = C.c_int64()
    assert lib.dc_debug_png_host(img.ctypes.data, 8, 8, 1, small.ctypes.data, small.size, C.byref(n), None, 0,
                                 None) == _lib.DC_EINVAL
    assert b"out_bytes" in lib.dc_last_error()
    with pytest.raises(TypeError):
        host(np.zeros((4, 4, 2), np.uint8))


def test_args_layout():
    from unet_dc_segmentation_b200 import _lib
    f = {name: getattr(_lib.PngArgs, name).offset for name, _ in _lib.PngArgs._fields_}
    # typedef struct { const uint8_t* images; int B, H, W, C; uint8_t* out; int64_t out_bytes; int64_t* offsets;
    #                  void* workspace; size_t workspace_bytes; } dc_png_args_t  (LP64)
    assert f == {"images": 0, "B": 8, "H": 12, "W": 16, "C": 20, "out": 24, "out_bytes": 32, "offsets": 40,
                 "workspace": 48, "workspace_bytes": 56}
    assert C.sizeof(_lib.PngArgs) == 64
