"""Drop-in boundary tests: libb200heif.so's heif_encoder_plugin / heif_decoder_plugin inside the UNMODIFIED reference
libheif (oracle/_ref/libheif_ref.so).  Runs in a child process (see oracle/refheif.py for why)."""
import ctypes as C
import json
import os
import subprocess
import sys

import pytest

from oracle import bindings as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
have_ref = os.path.exists(os.path.join(ob.REF, "libheif_ref.so")) and os.path.exists(os.path.join(ob.REF, "liboracle_plugin.so")) and ob.avcodec_dir()


def child(mode):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "plugin_child.py"), mode], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    return json.loads(line[7:])


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads and exports every symbol of include/b200_heif.h and include/b200_heif_plugin_abi.h."""
    import re
    lib = C.CDLL(os.path.join(ROOT, "libheif_b200", "libb200heif.so"))
    names = set()
    for hdr in ("b200_heif.h", "b200_heif_plugin_abi.h"):
        src = open(os.path.join(ROOT, "include", hdr)).read()
        names |= set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", src))
    names -= {"b200_planes", "b200_geometry", "b200_color_options"}
    names |= {"plugin_info", "b200_encoder_plugin_info"}
    missing = [n for n in sorted(names) if not hasattr(lib, n)]
    assert not missing, missing


def test_abi_mirror_matches_reference_headers(tmp_path):
    """Sizes, member offsets and constants of include/b200_heif_plugin_abi.h equal those of the reference's own headers
    (tests/golden/abi_layout.txt: tests/abi/abi_layout.cc built with -DREFERENCE_HEADERS against them)."""
    exe = tmp_path / "abi_layout"
    r = subprocess.run(["g++", "-std=c++17", os.path.join(ROOT, "tests", "abi", "abi_layout.cc"), "-o", str(exe)],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]
    got = subprocess.run([str(exe)], stdout=subprocess.PIPE, text=True, check=True).stdout.splitlines()
    with open(os.path.join(ROOT, "tests", "golden", "abi_layout.txt")) as f:
        want = f.read().splitlines()
    assert got == want, [(g, w) for g, w in zip(got, want) if g != w]


@pytest.mark.skipif(not have_ref, reason="oracle/_ref reference build not present")
def test_encoder_plugin_through_reference_libheif():
    """heif_context_encode_image / heif_context_encode_grid drive our heif_encoder_plugin; the files decode with the CPU plugin."""
    res = child("encode-cpu")
    assert res["single_shape"] == [136, 600]
    assert res["grid_shape"] == [256, 1152]
    assert res["single_psnr_luma_vs_green"] > 18      # G is only a proxy for Y: this guards against gross corruption
    # oracle/heic_writer.py (used by the reference arm of bench.py) produces files the reference reads identically
    assert res["grid_md5_own_writer"] == res["grid_md5_cpu"]
    assert res["single_own_shape"] == [128, 384]


@pytest.mark.gpu
@pytest.mark.skipif(not have_ref, reason="oracle/_ref reference build not present")
def test_decoder_plugin_drop_in_bit_exact(cuda):
    """heif_decode_image() of the unmodified reference with our decoder plugin == with the CPU (FFmpeg) plugin, bit for bit,
    for a single image and for a grid decoded from 8 libheif threads (one plugin instance per tile)."""
    res = child("roundtrip-gpu")
    assert res["single_md5_gpu"] == res["single_md5_cpu"]
    assert res["grid_md5_gpu"] == res["grid_md5_cpu"]
    assert res["single_md5_default"] == res["single_md5_cpu"] and res["grid_md5_default"] == res["grid_md5_cpu"]
    # sequence call order (SURVEY 8f N4, intra-only): one picture per push_data2, user_data echoed in order, parameter sets reused
    assert res["sequence_users"] == [1000, 1001, 1002] and res["sequence_planes_ok"] and res["sequence_drained"]


@pytest.mark.gpu
@pytest.mark.skipif(not have_ref, reason="oracle/_ref reference build not present")
def test_plugin_path_loading_and_concurrent_instances(cuda):
    """The reference loads libb200heif.so through LIBHEIF_PLUGIN_PATH (dlopen + `plugin_info`, plugins_unix.cc:103-119) and
    decodes with it, bit-exact; 64 plugin instances in flight at once (heif_context_set_max_decoding_threads(64) on an 8x8
    grid) go through the submission queue in batches and stay bit-exact; so do 16 different pictures decoded from 16 threads."""
    res = child("plugin-path-gpu")
    assert res["single_md5_gpu"] == res["single_md5_cpu"]
    assert res["grid_md5_gpu"] == res["grid_md5_cpu"]
    for rep in range(3):
        assert res[f"grid64_md5_gpu_{rep}"] == res["grid64_md5_cpu"]
    assert res["queue_max_batch"] > 1, res            # concurrent calls were really batched
    assert res["mixed_ok"], res.get("mixed_bad")
    assert res["chroma_formats_ok"], res.get("chroma_formats_bad")      # 4:2:2 / 4:4:4 items through heif_decode_image
