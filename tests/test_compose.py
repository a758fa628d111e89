"""Overlay compositing (SURVEY 8 a11) and nearest-neighbour scaling (a12).

CPU: the C restatement (oracle/color_oracle.c) against the UNMODIFIED reference (HeifPixelImage::overlay /
scale_nearest_neighbor, libheif/image/pixelimage.cc:1637-1972), whose results are stored in
tests/golden/reference_outputs.json (util.reference_fingerprint).
GPU: the CUDA kernels (libheif_b200/csrc/b200_compose.cu) against the restatement, bit-exact.
"""
import os
import numpy as np
import pytest

from util import fingerprint, reference_fingerprint

OVERLAY_CASES = [
    # (canvas w, h, background, [(child w, h, alpha?, dx, dy), ...])
    (64, 48, (0x1234, 0x8000, 0xffff, 0xffff), [(16, 16, False, 4, 5)]),
    (64, 48, (0, 0, 0, 0), [(32, 24, True, 10, 3), (20, 20, False, 50, 40)]),          # second child clipped right / bottom
    (40, 30, (0x8080, 0x4040, 0x2020, 0), [(25, 25, False, -7, -9)]),                   # negative offsets, copy path (reference loop bounds)
    (40, 30, (0x8080, 0x4040, 0x2020, 0), [(25, 25, True, -7, -9)]),                    # negative offsets, alpha path
    (40, 30, (0xffff, 0, 0, 0), [(100, 80, True, -30, -20)]),                           # child larger than the canvas
    (33, 17, (0x0100, 0x0200, 0x0300, 0), [(8, 8, True, 40, 2), (8, 8, False, -8, 0), (5, 5, True, 32, 16)]),   # outside right, outside left, 1-px overlap
    (50, 50, (0, 0xffff, 0, 0), [(50, 50, True, 0, 0), (10, 60, True, 45, -5)]),
]


def _children(spec, seed):
    rng = np.random.default_rng(seed)
    out = []
    for (w, h, alpha, dx, dy) in spec:
        rgb = rng.integers(0, 256, (3, h, w), dtype=np.uint8)
        al = rng.integers(0, 256, (h, w), dtype=np.uint8) if alpha else None
        if al is not None:
            al[::3, ::2] = 255; al[1::4, 1::3] = 0
        out.append((rgb, al, dx, dy))
    return out


SCALE_CASES = [
    # (colorspace, chroma, bpp, w, h, ow, oh, alpha)   colorspace 0 YCbCr, 1 RGB planar, 2 mono, 3 interleaved
    (0, 1, 8, 64, 48, 32, 24, False),
    (0, 1, 8, 31, 17, 64, 40, True),       # odd sizes up, with alpha (the alpha-plane-to-image-size use of SURVEY a12)
    (0, 2, 10, 40, 20, 13, 33, False),
    (0, 3, 12, 16, 16, 50, 7, False),
    (1, 3, 8, 20, 30, 45, 11, True),
    (2, 0, 8, 9, 9, 4, 20, False),
    (3, 10, 8, 24, 10, 17, 23, False),     # interleaved RGB
    (3, 11, 8, 24, 10, 40, 5, False),      # interleaved RGBA
]


def _scale_planes(cs, chroma, bpp, w, h, alpha, seed):
    rng = np.random.default_rng(seed)
    dt = np.uint8 if bpp <= 8 else np.uint16
    hi = 1 << bpp
    if cs == 3:
        comps = 3 if chroma == 10 else 4
        return [rng.integers(0, hi, (h, w * comps)).astype(dt)], [comps]
    sh = 1 if chroma in (1, 2) else 0
    sv = 1 if chroma == 1 else 0
    shapes = {0: [(h, w), ((h + sv) >> sv, (w + sh) >> sh), ((h + sv) >> sv, (w + sh) >> sh)], 1: [(h, w)] * 3, 2: [(h, w)]}[cs]
    if alpha:
        shapes = shapes + [(h, w)]
    return [rng.integers(0, hi, s).astype(dt) for s in shapes], [1] * len(shapes)


def _out_plane_sizes(cs, chroma, ow, oh, nplanes, alpha):
    if cs == 3 or cs == 1 or cs == 2:
        return [(ow, oh)] * nplanes
    sh = 1 if chroma in (1, 2) else 0
    sv = 1 if chroma == 1 else 0
    sizes = [(ow, oh), ((ow + sh) >> sh, (oh + sv) >> sv), ((ow + sh) >> sh, (oh + sv) >> sv)]
    return sizes + ([(ow, oh)] if alpha else [])


@pytest.mark.parametrize("case", range(len(OVERLAY_CASES)))
def test_overlay_oracle_matches_reference(case):
    from oracle import bindings as ob
    cw, ch, bkg, spec = OVERLAY_CASES[case]
    kids = _children(spec, 100 + case)
    got = ob.oracle_overlay(cw, ch, bkg, kids)
    assert fingerprint(got) == reference_fingerprint("ref_overlay", cw, ch, bkg, kids)


@pytest.mark.parametrize("case", range(len(SCALE_CASES)))
def test_scale_oracle_matches_reference(case):
    from oracle import bindings as ob
    cs, chroma, bpp, w, h, ow, oh, alpha = SCALE_CASES[case]
    planes, comps = _scale_planes(cs, chroma, bpp, w, h, alpha, 200 + case)
    sizes = _out_plane_sizes(cs, chroma, ow, oh, len(planes), alpha)
    got = np.concatenate([ob.oracle_scale_plane(p, sw, sh_, (w, h), (ow, oh), c).reshape(-1).view(np.uint8) for p, c, (sw, sh_) in zip(planes, comps, sizes)])
    assert fingerprint(got) == reference_fingerprint("ref_scale_nn", cs, chroma, bpp, planes, w, h, ow, oh, alpha)


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(OVERLAY_CASES)))
def test_overlay_gpu_matches_oracle(case):
    import torch
    import libheif_b200 as lb
    from oracle import bindings as ob
    cw, ch, bkg, spec = OVERLAY_CASES[case]
    kids = _children(spec, 100 + case)
    want = ob.oracle_overlay(cw, ch, bkg, kids)
    canvas = lb.compose.overlay_canvas(cw, ch, bkg)
    for rgb, al, dx, dy in kids:
        lb.compose.overlay(canvas, torch.from_numpy(rgb).cuda(), dx, dy, None if al is None else torch.from_numpy(al).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(canvas.cpu().numpy(), want)


@pytest.mark.gpu
def test_overlay_gpu_large_canvas():
    """4096 x 3072 canvas, three 2048 x 2048 children (one blended): property = equality with the restatement."""
    import torch
    import libheif_b200 as lb
    from oracle import bindings as ob
    spec = [(2048, 2048, False, 0, 0), (2048, 2048, True, 1500, 700), (2048, 2048, True, -100, 2000)]
    kids = _children(spec, 7)
    want = ob.oracle_overlay(4096, 3072, (0x4000, 0x8000, 0xc000, 0), kids)
    canvas = lb.compose.overlay_canvas(4096, 3072, (0x4000, 0x8000, 0xc000, 0))
    for rgb, al, dx, dy in kids:
        lb.compose.overlay(canvas, torch.from_numpy(rgb).cuda(), dx, dy, None if al is None else torch.from_numpy(al).cuda())
    assert np.array_equal(canvas.cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(SCALE_CASES)))
def test_scale_gpu_matches_oracle(case):
    import torch
    import libheif_b200 as lb
    from oracle import bindings as ob
    cs, chroma, bpp, w, h, ow, oh, alpha = SCALE_CASES[case]
    planes, comps = _scale_planes(cs, chroma, bpp, w, h, alpha, 200 + case)
    sizes = _out_plane_sizes(cs, chroma, ow, oh, len(planes), alpha)
    for p, c, (sw, sh_) in zip(planes, comps, sizes):
        want = ob.oracle_scale_plane(p, sw, sh_, (w, h), (ow, oh), c)
        t = torch.from_numpy(p.view(np.int16) if p.dtype == np.uint16 else p).cuda()
        got = lb.compose.scale_nearest_plane(t, sw, sh_, (w, h), (ow, oh), c).cpu().numpy()
        if p.dtype == np.uint16:
            got = got.view(np.uint16)
        assert np.array_equal(got, want)
