"""CPU: pin the colour restatement (oracle/color_oracle.c) against the UNMODIFIED reference
(HeifPixelImage transforms + convert_colorspace) on LCG-random planes; the reference's results are stored in
tests/golden/reference_outputs.json (util.reference_fingerprint).
Mirrors the differential strategy of the reference's tests/conversion.cc (every state pair, small images)."""
import numpy as np
import pytest

from util import fingerprint, oracle_postprocess, random_ycbcr, reference_fingerprint

SIZES = [(2, 2), (6, 4), (34, 18), (64, 64), (130, 70)]
CASES = [
    # chroma, bpp, nclx (cp,tc,mc,full), out_chroma
    (1, 8, (1, 13, 6, 1), 10), (1, 8, (1, 13, 6, 0), 10), (1, 8, (2, 2, 2, 0), 10), (1, 8, (1, 13, 1, 0), 10),
    (1, 8, (9, 16, 9, 0), 10), (1, 8, (1, 13, 5, 1), 11), (1, 8, (1, 13, 6, 0), 11), (1, 8, None, 10),
    (3, 8, (1, 13, 6, 1), 10), (3, 8, (1, 13, 6, 0), 10), (2, 8, (1, 13, 6, 1), 10), (2, 8, (1, 13, 1, 0), 11),
    (1, 10, (9, 16, 9, 0), 14), (1, 10, (9, 16, 9, 1), 14), (1, 12, (9, 16, 9, 0), 14), (1, 10, (9, 16, 9, 0), 12),
    (1, 10, (1, 13, 1, 0), 10), (1, 12, (1, 13, 6, 1), 10), (1, 8, (1, 13, 6, 0), 3), (1, 10, (9, 16, 9, 0), 3),
    (1, 8, (1, 13, 12, 1), 10), (1, 8, (9, 13, 13, 0), 10), (1, 8, (1, 13, 4, 0), 10), (1, 8, (1, 13, 7, 1), 10),
]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("size", SIZES)
def test_restatement_matches_reference(case, size):
    chroma, bpp, nclx, outc = case
    w, h = size
    y, cb, cr, _ = random_ycbcr(0xB200 + w * 131 + h, w, h, chroma, bpp)
    hdr8 = 1 if (bpp > 8 and outc in (10, 11)) else 0
    got = oracle_postprocess(y, cb, cr, None, chroma, bpp, nclx, [], outc)
    assert fingerprint(*got) == reference_fingerprint("ref_postprocess", y, cb, cr, None, chroma, bpp, nclx, [], outc, hdr_to_8bit=hdr8)


@pytest.mark.parametrize("alpha_out", [10, 11])
@pytest.mark.parametrize("nclx", [(1, 13, 6, 1), (1, 13, 6, 0)])
def test_alpha_plane(alpha_out, nclx):
    y, cb, cr, a = random_ycbcr(77, 36, 20, 1, 8, alpha=True)
    got = oracle_postprocess(y, cb, cr, a if alpha_out == 11 else None, 1, 8, nclx, [], alpha_out)
    assert fingerprint(*got) == reference_fingerprint("ref_postprocess", y, cb, cr, a, 1, 8, nclx, [], alpha_out)


GEOM = [[(1, 90)], [(1, 180)], [(1, 270)], [(2, 0)], [(2, 1)], [(3, 2, 21, 4, 17)], [(1, 90), (2, 1)],
        [(3, 4, 27, 2, 13), (1, 270)], [(2, 0), (1, 90), (3, 0, 9, 0, 15)]]


@pytest.mark.parametrize("ops", GEOM)
@pytest.mark.parametrize("fmt", [(1, 8, (1, 13, 6, 0), 10), (1, 10, (9, 16, 9, 0), 14), (3, 8, (1, 13, 6, 1), 11)])
def test_geometry_then_colour(ops, fmt):
    chroma, bpp, nclx, outc = fmt
    y, cb, cr, _ = random_ycbcr(1234, 32, 24, chroma, bpp)
    got = oracle_postprocess(y, cb, cr, None, chroma, bpp, nclx, ops, outc)
    assert fingerprint(*got) == reference_fingerprint("ref_postprocess", y, cb, cr, None, chroma, bpp, nclx, ops, outc)


def test_bilinear_golden_table_of_reference_tests():
    """tests/conversion.cc:697-724 ('Bilinear upsampling'): Cb {10,40;100,240}, Cr {255,200;50,0} -> 4x4 tables."""
    import ctypes as C
    from oracle import bindings as ob
    l = ob.lib()
    for src, want in (([10, 40, 100, 240], [10, 18, 33, 40, 33, 47, 76, 90, 78, 106, 162, 190, 100, 135, 205, 240]),
                      ([255, 200, 50, 0], [255, 241, 214, 200, 204, 190, 163, 150, 101, 88, 63, 50, 50, 38, 13, 0])):
        a = np.array(src, np.uint16); out = np.zeros(16, np.uint16)
        l.co_bilinear_420_to_444(a.ctypes.data_as(C.c_void_p), 4, 4, out.ctypes.data_as(C.c_void_p))
        assert out.tolist() == want


BILINEAR_CASES = [(1, 8, (1, 13, 6, 0), 10), (1, 8, (1, 13, 6, 1), 10), (1, 8, (1, 13, 1, 0), 11), (1, 10, (9, 16, 9, 0), 14), (1, 12, (9, 16, 9, 1), 14)]


@pytest.mark.parametrize("case", BILINEAR_CASES)
@pytest.mark.parametrize("size", [(4, 4), (6, 4), (34, 18), (33, 17), (64, 64), (130, 70)])
def test_bilinear_pipeline_matches_reference(case, size):
    """heif-dec -C bilinear: only_use_preferred_chroma_algorithm=1 (SURVEY F6), incl. the border indexing of the reference."""
    chroma, bpp, nclx, outc = case
    w, h = size
    y, cb, cr, _ = random_ycbcr(0xB200 + w * 7 + h, w, h, chroma, bpp)
    got = oracle_postprocess(y, cb, cr, None, chroma, bpp, nclx, [], outc, bilinear=1)
    assert fingerprint(*got) == reference_fingerprint("ref_postprocess", y, cb, cr, None, chroma, bpp, nclx, [], outc, only_preferred=1, upsampling=2)


# 4:4:4 conversion point of the reference (pixelimage.cc:1187-1215, 1370-1396, 1458-1481): 4:2:0 pictures with an odd
# crop origin / odd sizes under rotate or mirror are first converted to 4:4:4 (bilinear; limited-range pictures are also
# range-converted through RGB because the conversion's target profile is full range).
DETOUR = [
    (34, 18, [(3, 3, 30, 1, 16)]),                                # crop with odd left and top
    (34, 18, [(3, 2, 30, 1, 16)]),                                # odd top only
    (33, 18, [(1, 90)]), (34, 17, [(1, 270)]), (33, 17, [(1, 180)]),
    (33, 18, [(2, 1)]), (34, 17, [(2, 0)]),
    (64, 48, [(3, 2, 61, 2, 45), (3, 1, 50, 0, 40)]),             # even crop, then odd crop of the result
    (64, 48, [(1, 90), (3, 2, 40, 3, 50), (2, 0), (1, 180)]),     # rotate, odd crop, then more transforms on the 4:4:4 picture
    (63, 47, [(1, 180), (3, 5, 40, 3, 30)]),
]


@pytest.mark.parametrize("case", DETOUR)
@pytest.mark.parametrize("fmt", [(8, (1, 13, 6, 1), 10, False), (8, (1, 13, 6, 1), 11, True), (10, (9, 16, 9, 1), 14, False), (12, (1, 13, 1, 1), 10, False),
                                 # limited range: the conversion point also range-converts, through RGB (restated in the oracle; the CUDA path refuses these)
                                 (8, (1, 13, 6, 0), 10, False), (8, (2, 2, 2, 0), 11, True), (10, (9, 16, 9, 0), 14, False), (12, (1, 13, 1, 0), 3, False)])
def test_444_detour_matches_reference(case, fmt):
    w, h, ops = case
    bpp, nclx, outc, alpha = fmt
    y, cb, cr, a = random_ycbcr(77, w, h, 1, bpp, alpha=alpha)
    got = oracle_postprocess(y, cb, cr, a, 1, bpp, nclx, ops, outc)
    assert fingerprint(*got) == reference_fingerprint("ref_postprocess", y, cb, cr, a, 1, bpp, nclx, ops, outc)


@pytest.mark.parametrize("ops", GEOM[:6])
def test_bilinear_after_geometry_matches_reference(ops):
    """only_use_preferred_chroma_algorithm + bilinear: the upsampling op sees the picture AFTER rotate / mirror / crop."""
    y, cb, cr, _ = random_ycbcr(99, 32, 24, 1, 8)
    got = oracle_postprocess(y, cb, cr, None, 1, 8, (1, 13, 6, 0), ops, 10, bilinear=1)
    assert fingerprint(*got) == reference_fingerprint("ref_postprocess", y, cb, cr, None, 1, 8, (1, 13, 6, 0), ops, 10, only_preferred=1, upsampling=2)


# matrix_coefficients 0 (GBR), 8 (YCgCo), 16 (YCgCo-Re): special branches of the generic op; the dedicated 4:2:0 ops ignore
# them (16) or are not selected (0, 8).  Restated in the oracle for round 2; the CUDA path still refuses these matrices.
@pytest.mark.parametrize("mc", [0, 8, 16])
@pytest.mark.parametrize("chroma", [1, 2, 3])
@pytest.mark.parametrize("bpp,outc", [(8, 10), (8, 11), (8, 3), (10, 10), (10, 14), (10, 3), (12, 15)])
@pytest.mark.parametrize("full", [0, 1])
def test_special_matrices_match_reference(mc, chroma, bpp, outc, full):
    y, cb, cr, a = random_ycbcr(4242 + mc, 34, 18, chroma, bpp, alpha=outc in (11, 15))
    got = oracle_postprocess(y, cb, cr, a, chroma, bpp, (1, 13, mc, full), [], outc)
    assert fingerprint(*got) == reference_fingerprint("ref_postprocess", y, cb, cr, a, chroma, bpp, (1, 13, mc, full), [], outc)


# 4:2:2 pictures: rotate 90 / 270 always, 180 with odd height, horizontal mirror with odd width and crop with odd left
# convert to 4:4:4 first (Op_YCbCr422_bilinear_to_YCbCr444).  Restated for round 2; the CUDA path refuses these chains.
DETOUR_422 = [
    (34, 18, [(1, 90)]), (33, 18, [(1, 270)]), (34, 17, [(1, 180)]), (34, 18, [(1, 180)]),
    (33, 17, [(2, 1)]), (34, 17, [(2, 0)]), (64, 48, [(3, 3, 61, 1, 45), (1, 90)]), (64, 48, [(3, 2, 61, 1, 45)]),
]


@pytest.mark.parametrize("case", DETOUR_422)
@pytest.mark.parametrize("fmt", [(8, (1, 13, 6, 1), 10, False), (8, (1, 13, 6, 0), 11, True), (10, (9, 16, 9, 0), 14, False), (12, (1, 13, 1, 1), 3, False)])
def test_444_detour_422_matches_reference(case, fmt):
    w, h, ops = case
    bpp, nclx, outc, alpha = fmt
    y, cb, cr, a = random_ycbcr(78, w, h, 2, bpp, alpha=alpha)
    got = oracle_postprocess(y, cb, cr, a, 2, bpp, nclx, ops, outc)
    assert fingerprint(*got) == reference_fingerprint("ref_postprocess", y, cb, cr, a, 2, bpp, nclx, ops, outc)


# ---- encoder-side direction: Op_RGB24_32_to_YCbCr (rgb2yuv.cc:575-808) ----
RGB2YCC_SIZES = [(1, 1), (2, 2), (3, 3), (5, 4), (4, 5), (16, 16), (33, 17), (64, 48)]
RGB2YCC_NCLX = [(1, 13, 6, 1), (1, 13, 6, 0), (1, 13, 1, 1), (1, 13, 1, 0), (9, 16, 9, 0), (9, 16, 9, 1), (1, 13, 5, 1), (2, 2, 2, 0), (2, 2, 2, 1),
                (1, 13, 12, 1), (9, 13, 13, 0), (1, 13, 4, 0), (1, 13, 7, 1)]


def rgb_pattern(seed, w, h, bpp):
    """LCG bytes with saturated corners and flat runs (clipping and rounding ties are where restatements go wrong)."""
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (h, w * bpp), dtype=np.uint8)
    img[0, :bpp] = 255
    img[-1, -bpp:] = 0
    if w >= 4:
        img[h // 2, : 2 * bpp] = np.tile(np.array([255, 0, 0, 128][:bpp], np.uint8), 2)
    return img


@pytest.mark.parametrize("size", RGB2YCC_SIZES)
@pytest.mark.parametrize("alpha", [0, 1])
@pytest.mark.parametrize("out_chroma", [1, 2, 3])
def test_rgb_to_ycbcr_restatement_matches_reference(size, alpha, out_chroma):
    from oracle.bindings import oracle_rgb_to_ycbcr
    w, h = size
    rgb = rgb_pattern(0x5EED + w * 977 + h * 31 + alpha, w, h, 4 if alpha else 3)
    for nclx in RGB2YCC_NCLX:
        got = oracle_rgb_to_ycbcr(rgb, alpha, out_chroma, nclx)
        assert fingerprint(got) == reference_fingerprint("ref_rgb_to_ycbcr", rgb, alpha, out_chroma, nclx), f"Y, Cb, Cr or A differs for nclx {nclx}"
