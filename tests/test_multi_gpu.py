"""Multi-GPU parity on hardware (skipped with fewer than 2 devices): bench.py's sharded decode of a grid on 2 GPUs must give
the same bytes as on 1 GPU, and both must match what the unmodified reference decodes (bench.py's own in-run check)."""
import json
import os
import subprocess
import sys

import pytest

from oracle import bindings as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# md5 of the RGB24 heif_decode_image of the unmodified reference (CPU decoder plugin) returns for the 4 x 4 grid of bench
# tiles run_bench decodes: `python -m oracle.ref_arm --side 4 --sub 4` prints it as rgb_md5
REFERENCE_RGB_MD5_4X4 = "1c31ae3b1f537bac349d093950bfc0df"
# bench.py compares with the reference in the run where the reference build exists
have_ref = bool(os.path.exists(os.path.join(ob.REF, "libheif_ref.so")) and os.path.exists(os.path.join(ob.REF, "liboracle_plugin.so")) and ob.avcodec_dir())


def run_bench(n, port):
    base = ["bench.py", "--gpus", str(n), "--steps", "1", "--warmup", "1", "--tiles-side", "4", "--ref-sample-side", "4", "--no-ctb64", "--no-plugin-leg"]
    cmd = [sys.executable] + base if n == 1 else [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
                                                  "--master-port", str(port)] + base
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])


@pytest.mark.gpu
def test_two_gpus_equal_one_gpu_equal_reference(cuda):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    one = run_bench(1, 29631)
    two = run_bench(2, 29632)
    assert one["rgb_md5"] == two["rgb_md5"] == REFERENCE_RGB_MD5_4X4
    assert one["parity_checked"] == two["parity_checked"] == have_ref, (one.get("parity"), two.get("parity"))
    assert two["n_gpus"] == 2


@pytest.mark.gpu
def test_bench_checks_itself_against_the_reference(cuda):
    """1 GPU: the bench's RGB is what heif_decode_image of the unmodified reference returns (stored md5), and where the
    reference build exists the bench line carries parity_checked = true from its own in-run comparison."""
    one = run_bench(1, 29633)
    assert one["rgb_md5"] == REFERENCE_RGB_MD5_4X4
    if have_ref:
        assert one["parity_checked"] is True, one.get("parity")
        assert one["parity"]["mismatching_bytes"] == 0


def run_config5(n, port, dump):
    base = [os.path.join("scripts", "config5_bench.py"), "--tile", "256", "--ntiles", "12", "--grid", "8", "--steps", "1", "--warmup", "1", "--dump-dir", dump]
    cmd = [sys.executable] + base if n == 1 else [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
                                                  "--master-port", str(port)] + base
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])


@pytest.mark.gpu
def test_config5_region_of_interest_round_robin(cuda, tmp_path):
    """BASELINE config 5 (scaled down: 12 LCG-picked 256x256 12-bit tiles of an 8x8 grid): every tile's RRGGBB_LE equals the
    oracle (restatement planes + colour oracle); with 2 GPUs the round-robin sharded run gives the same bytes."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import config5_bench as c5
    from oracle import bindings as ob
    from util import oracle_postprocess
    d1 = tmp_path / "one"; d1.mkdir()
    one = run_config5(1, 29641, str(d1))
    picks = c5.picks_lcg(12, 64)
    for t in picks[:4]:
        au = c5.make_tile(t, 256, 12)
        planes, info = ob.restatement_decode(au)
        want, ow, oh = oracle_postprocess(planes[0], planes[1], planes[2], None, 1, 12, (info["cp"], info["tc"], info["mc"], info["full_range"]), [], 14)
        got = np.fromfile(d1 / f"tile_{t}.rgb", dtype=np.uint8)
        assert (ow, oh) == (256, 256) and np.array_equal(got, want), f"tile {t}"
    if torch.cuda.device_count() >= 2:
        d2 = tmp_path / "two"; d2.mkdir()
        two = run_config5(2, 29642, str(d2))
        assert two["n_gpus"] == 2 and two["md5_of_tile_md5s"] == one["md5_of_tile_md5s"]
