"""CPU: pin the C restatement of HEVC intra decoding (oracle/hevc_oracle.c) on an independent conforming decoder
(FFmpeg libavcodec, oracle/ffhevc.c) for the reference's fixtures and for every synthetic stream; plus the golden md5s
of SURVEY.md Appendix C for the reference fixtures (planes of examples/example.heic)."""
import hashlib
import os

import numpy as np
import pytest

from hevc_cases import all_streams, cpu_extra_streams, synth_params, synth_source, synth_stream
from oracle import bindings as ob

have_ffmpeg = ob.avcodec_dir() is not None

# FFmpeg 62's chroma SAO reads neighbours whose horizontal-edge deblocking is still deferred when log2_ctb_size == 4
# (its deblocking defers chroma horizontal edges by 16 luma samples = one whole 16x16 CTB), so it deviates from H.265
# 8.7.3 ("deblocked sample array") at a handful of CTB-corner chroma samples.  Those streams are pinned on luma +
# the no-SAO / no-deblocking variants instead.
FFMPEG_CTB16_CHROMA_SAO = {"ctb16_basic"}


def ffmpeg_planes(name, nplanes):
    """Planes of stream `name` FFmpeg 62 decodes per H.265.  Two more deviations of that build, both established on LOSSLESS
    streams (every coding unit cu_transquant_bypass: the decoded picture must equal the encoder's input, which the
    restatement reproduces on all planes and FFmpeg only on luma, test_lossless_streams_reproduce_their_source):
      * with SAO enabled, FFmpeg's chroma SAO does not leave the samples of cu_transquant_bypass units / of PCM units under
        pcm_loop_filter_disabled_flag unchanged (8.7.3 requires SaoTypeIdx to be treated as 0 there): luma only, the
        chroma path is pinned by the sao=0 variants of the same streams (x_*_nosao);
      * 4:0:0 streams with PCM units lose CABAC synchronisation in FFmpeg ("cu_qp_delta ... outside the valid range"): not compared."""
    if name in FFMPEG_CTB16_CHROMA_SAO:
        return [0]
    p = synth_params(name)
    if p is not None:
        o = p[5]
        if o.get("pcm") and not p[4]:
            return []
        if p[4] == 2 and o.get("log2_ctb_size") == 4 and o.get("sao", 1):
            return [0]                                     # the CTB-16 chroma SAO deviation above, 4:2:2
        if o.get("sao", 1) and (o.get("transquant_bypass") or o.get("pcm") == 2):
            return [0]
    return list(range(nplanes))


@pytest.mark.skipif(not have_ffmpeg, reason="FFmpeg (cv2 wheel) not present")
@pytest.mark.parametrize("name,au", all_streams() + cpu_extra_streams(), ids=[s[0] for s in all_streams() + cpu_extra_streams()])
def test_restatement_matches_ffmpeg(name, au):
    ff, bd, ch = ob.ffmpeg_decode(au)
    rs, info = ob.restatement_decode(au)
    assert info["bit_depth"] == bd and info["chroma"] == ch
    for c in ffmpeg_planes(name, len(ff)):
        assert np.array_equal(ff[c], rs[c]), f"plane {c} differs at {np.argwhere(ff[c] != rs[c])[:3].tolist()}"


LOSSLESS = [s[0] for s in __import__("hevc_cases").SYNTH + __import__("hevc_cases").SYNTH_CPU_EXTRA if s[5].get("transquant_bypass") == 2]


@pytest.mark.parametrize("name", LOSSLESS)
def test_lossless_streams_reproduce_their_source(name):
    """cu_transquant_bypass on every coding unit: scaling, transform and all in-loop filters are bypassed (8.6.2, 8.7.2.5.7,
    8.7.3), so the decoded picture IS the picture that was encoded -- a pin of the bypass path that needs no second decoder."""
    rs, info = ob.restatement_decode(synth_stream(name))
    src = synth_source(name)
    for c in range(len(rs)):
        assert np.array_equal(rs[c], src[c]), f"plane {c}"


def test_example_heic_golden_md5():
    """SURVEY.md Appendix C: FFmpeg planes of examples/example.heic item 20004."""
    au = dict(all_streams())["example_primary_1280x854.au"]
    rs, _ = ob.restatement_decode(au)
    md5 = [hashlib.md5(p.astype(np.uint8).tobytes()).hexdigest() for p in rs]
    assert md5 == ["5a0423057f3fede64a297243982465c7", "8a2344a26a2347f045842be7f731085c", "29ad6bcbe5dd90a536d0abe36777a1b5"]


# md5 of every access unit the unmodified reference libheif pushes into a decoder plugin while it decodes its own fixture
# files, as `tests/golden/make_streams.py --check` prints them
REFERENCE_STREAM_MD5 = {
    "example_primary_1280x854": "00e077c93335db561337ae4e14312b4d",
    "rainbow_452x462": "fb9b9131bd5e8861b97590d9d5b1d295",
    "hevc32_64x64": "05d5015c145ee9e3d3829acbb2249a3e",
    "colors_alpha_main_64x64": "dc8a95d38eabb2c8a90d5264be76a0ef",
    "colors_alpha_aux_64x64": "141d2c752979453eadebb364b2e813ab",
    "colors_noalpha_64x64": "dc8a95d38eabb2c8a90d5264be76a0ef",
}


def test_golden_streams_are_what_the_reference_pushes_into_a_decoder_plugin():
    """tests/golden/streams/*.au are byte-for-byte what the unmodified reference libheif pushes into a decoder plugin for
    the reference's fixture files (tests/golden/make_streams.py regenerates them from the reference)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for name, md5 in REFERENCE_STREAM_MD5.items():
        with open(os.path.join(root, "tests", "golden", "streams", name + ".au"), "rb") as f:
            assert hashlib.md5(f.read()).hexdigest() == md5, name
