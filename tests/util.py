"""Shared helpers for the test-suite (test infrastructure; may import oracle/)."""
import atexit
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import bindings as ob  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
REFERENCE_OUTPUTS = os.path.join(GOLDEN, "reference_outputs.json")


def _feed(h, v):
    if isinstance(v, np.ndarray):
        h.update(f"a{v.dtype.str}{v.shape};".encode())
        h.update(np.ascontiguousarray(v).tobytes())
    elif isinstance(v, (list, tuple)):
        h.update(b"(")
        for x in v:
            _feed(h, x)
        h.update(b")")
    else:
        h.update(f"{v!r};".encode())


def fingerprint(*parts):
    """Digest of dtype, shape and bytes of every array in parts (and of every other value by repr): equal fingerprints
    mean np.array_equal on every array and equality of everything else."""
    h = hashlib.sha256()
    _feed(h, parts)
    return h.hexdigest()[:32]


_stored = None


def _write_reference_outputs():
    with open(REFERENCE_OUTPUTS, "w") as f:
        json.dump(dict(sorted(_stored.items())), f, indent=0)
        f.write("\n")


def _reference_outputs():
    global _stored
    if _stored is None:
        if os.environ.get("B200_RECORD_REFERENCE"):
            _stored = {}
            atexit.register(_write_reference_outputs)
        else:
            with open(REFERENCE_OUTPUTS) as f:
                _stored = json.load(f)
    return _stored


def reference_fingerprint(name, *args, **kw):
    """fingerprint() of what the unmodified reference libheif returns for oracle.bindings.<name>(*args, **kw): for
    ref_postprocess the output bytes, width and height; for the others the whole result.

    The fingerprints are stored in tests/golden/reference_outputs.json, keyed by a digest of the call, so the comparison
    with the reference runs wherever the tests run.  Where the reference build (oracle/_ref) exists, the reference is also
    run and must agree with what is stored; with B200_RECORD_REFERENCE=1 its results replace the file instead:
        B200_RECORD_REFERENCE=1 python -m pytest tests/test_color_oracle.py tests/test_compose.py -m "not gpu"
    """
    key = fingerprint(name, args, sorted(kw.items()))
    stored = _reference_outputs()
    if ob.ref_plugin() is not None:
        r = getattr(ob, name)(*args, **kw)
        fp = fingerprint(*(r[:3] if name == "ref_postprocess" else (r,)))
        if os.environ.get("B200_RECORD_REFERENCE"):
            stored[key] = fp
        else:
            assert stored.get(key) == fp, f"{name}: the reference build disagrees with tests/golden/reference_outputs.json"
        return fp
    assert key in stored, f"{name}: no stored reference output for this call (see util.reference_fingerprint)"
    return stored[key]


def lcg_plane(seed, h, w, lo, hi):
    """32-bit LCG s = s*1664525 + 1013904223 (SURVEY.md section 8d), vectorised by jumping ahead."""
    n = h * w
    out = np.empty(n, dtype=np.uint32)
    s = np.uint64(seed & 0xFFFFFFFF)
    a, c, m = 1664525, 1013904223, 1 << 32
    # sequential generation in chunks (python ints) is slow for big planes: use the closed form via numpy powers
    idx = np.arange(1, n + 1, dtype=np.uint64)
    # compute a^k and (a^k - 1)/(a - 1) * c mod 2^32 with repeated squaring over bits
    ak = np.ones(n, dtype=np.uint64)
    ck = np.zeros(n, dtype=np.uint64)
    base_a, base_c = np.uint64(a), np.uint64(c)
    mask = np.uint64(m - 1)
    k = idx.copy()
    while k.any():
        bit = (k & np.uint64(1)).astype(bool)
        ck = np.where(bit, (ck * base_a + base_c) & mask, ck)
        ak = np.where(bit, (ak * base_a) & mask, ak)
        base_c = (base_c * (base_a + np.uint64(1))) & mask
        base_a = (base_a * base_a) & mask
        k >>= np.uint64(1)
    out = ((ak * s + ck) & mask).astype(np.uint32)
    vals = lo + ((out >> np.uint32(8)) % np.uint32(hi - lo + 1))
    return vals.reshape(h, w).astype(np.uint16)


def random_ycbcr(seed, w, h, chroma, bpp, alpha=False, full_range_values=True):
    sh = 1 if chroma in (1, 2) else 0
    sv = 1 if chroma == 1 else 0
    maxv = (1 << bpp) - 1
    y = lcg_plane(seed, h, w, 0, maxv)
    cb = cr = None
    if chroma:
        cw, ch = (w + sh) >> sh, (h + sv) >> sv
        cb = lcg_plane(seed + 1, ch, cw, 0, maxv)
        cr = lcg_plane(seed + 2, ch, cw, 0, maxv)
    a = lcg_plane(seed + 3, h, w, 0, maxv) if alpha else None
    return y, cb, cr, a


from oracle.bindings import oracle_postprocess, ref_plugin, ref_postprocess  # noqa: E402,F401
