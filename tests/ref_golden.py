"""TEST INFRASTRUCTURE: what the compiled reference (oracle/_ref) computed for the tests that compare with it.

tests/golden/make_golden.py calls record_reference() of those test modules where oracle/_ref is built and stores the
results in tests/golden/ref_outputs.json.gz, so that the comparisons run wherever the tests run.  Arrays of more than
SMALL elements are stored as digests (dtype, shape and SHA-256 of the bytes), and logs of more than SMALL lines as their
line count and a digest of each block of SMALL lines; jpeg_cases.compare and lines_diff take either form."""
import functools
import gzip
import hashlib
import json
import os
from types import SimpleNamespace

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_outputs.json.gz")
SMALL = 64
DECODED_FIELDS = ("geom", "pix_y", "pix_cb", "pix_cr", "dib", "mcu_map", "dht_histo", "stats")


def digest(a):
    a = np.ascontiguousarray(a)
    return "%s%s:%s" % (a.dtype.str, list(a.shape), hashlib.sha256(a.tobytes()).hexdigest()[:32])


def arr(a):
    """An array in stored form: its values when small, else its digest."""
    if a is None:
        return None
    a = np.asarray(a)
    return a.tolist() if a.size <= SMALL else digest(a)


def same(want, got):
    """want: an array in stored form; got: the array the code under test produced."""
    if want is None or got is None:
        return want is None and got is None
    if isinstance(want, str):
        return digest(got) == want
    return np.array_equal(np.asarray(want), np.asarray(got))


def decoded(d):
    """A tests/oracle_util.Decoded in stored form."""
    r = {f: arr(getattr(d, f)) for f in DECODED_FIELDS}
    r["blk_dc"] = [arr(b) for b in d.blk_dc]
    r["nerr"] = int(d.nerr)
    return r


def colour_stats(s):
    """Oracle.colour_stats() in stored form."""
    return {k: (int(v) if k == "count" else arr(v)) for k, v in s.items()}


def _blocks(lines):
    return [hashlib.sha256("\n".join(lines[i:i + SMALL]).encode()).hexdigest()[:16] for i in range(0, len(lines), SMALL)]


def lines(ls):
    """Log lines in stored form."""
    return list(ls) if len(ls) <= SMALL else {"n": len(ls), "blocks": _blocks(ls)}


def lines_diff(want, got):
    """[] when the log lines `got` equal the stored `want`, else where they first differ."""
    if isinstance(want, list):
        return [] if want == got else [len(want), len(got)] + [(i, a, b) for i, (a, b) in enumerate(zip(want, got)) if a != b][:3]
    gb = _blocks(got)
    if want["n"] == len(got) and want["blocks"] == gb:
        return []
    k = next((i for i, (a, b) in enumerate(zip(want["blocks"], gb)) if a != b), min(len(gb), len(want["blocks"])))
    return [want["n"], len(got), f"first differing block of {SMALL} lines starts at line {k * SMALL}:"] + got[k * SMALL:(k + 1) * SMALL]


@functools.lru_cache(maxsize=1)
def _load():
    with gzip.open(PATH, "rt") as f:
        return json.load(f)


def get(key):
    """The stored value of `key` (a KeyError names a case make_golden.py has not recorded)."""
    return _load()[key]


def get_decoded(key):
    """A stored decode as an object with Decoded's fields (arrays as stored: values or digests)."""
    r = dict(get(key))
    r["blk_dc"] = tuple(r["blk_dc"])
    return SimpleNamespace(**r)


def save(values):
    with gzip.GzipFile(PATH, "wb", mtime=0) as f:
        f.write(json.dumps(values, sort_keys=True, separators=(",", ":")).encode())
