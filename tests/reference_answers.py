"""The answers of the unmodified reference (fpng v1.0.6, its trainer, its fpng_test harness, and the lodepng, stb_image, wuffs and
pvpng decoders it verifies with), recorded per test in tests/golden/reference_answers.json.gz, so that the tests that compare with
the reference run on machines that do not have it.

Replay (the default): every call returns what the reference returned when the answers were recorded.  Each answer is stored with
a digest of the call's inputs (the bytes of the image or file and every other argument): a call whose inputs the reference was not
asked fails the test, and so does a test that leaves recorded calls unmade.  Pixels and file bytes are not stored: the oracle
(oracle/fpng_oracle.c) recomputes them and they must have the recorded length and sha256 prefix, so a replayed answer is the
reference's answer or the test fails.

Record: with oracle/_ref built (oracle/Makefile) and FPNGB_RECORD_REFERENCE=<path>, the calls go to the real reference and the
answers of every test that ran are written to <path> at the end of the session, merged with tests/golden/reference_answers.json.gz:

    FPNGB_RECORD_REFERENCE=tests/golden/reference_answers.json.gz python -m pytest tests
"""
from __future__ import annotations

import atexit
import gzip
import hashlib
import json
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "reference_answers.json.gz")
RECORD = os.environ.get("FPNGB_RECORD_REFERENCE")

_answers = None


def digest(b) -> str:
    """length and sha256 prefix of bytes or of an array's bytes"""
    a = bytes(b) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b).tobytes()
    return f"{len(a)}:{hashlib.sha256(a).hexdigest()[:16]}"


def inputs_digest(*parts) -> str:
    """sha256 prefix of a call's inputs: bytes, arrays (their bytes), integers, strings and lists of integers"""
    h = hashlib.sha256()
    for p in parts:
        if isinstance(p, np.ndarray):
            b = np.ascontiguousarray(p).tobytes()
        elif isinstance(p, (bytes, bytearray)):
            b = bytes(p)
        elif isinstance(p, (list, tuple)):
            b = np.asarray(p, np.int64).tobytes()
        elif isinstance(p, (bool, int, np.integer)):
            b = str(int(p)).encode()
        else:
            b = str(p).encode()
        h.update(len(b).to_bytes(8, "little") + b)
    return h.hexdigest()[:12]


class Digest:
    """Bytes the reference produced and the oracle cannot recompute: equal to bytes of the same digest."""

    def __init__(self, d: str):
        self.d = d

    def __eq__(self, other):
        return isinstance(other, (bytes, bytearray, np.ndarray)) and digest(other) == self.d

    def __len__(self):
        return int(self.d.split(":")[0])

    def __repr__(self):
        return f"Digest({self.d!r})"


def _load() -> dict:
    global _answers
    if _answers is None:
        _answers = {}
        if os.path.exists(GOLDEN):
            with gzip.open(GOLDEN, "rt") as f:
                _answers = json.load(f)
        if RECORD:
            atexit.register(_save)
    return _answers


def _save():
    with open(RECORD, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as gz:
        lines = (f"{json.dumps(k)}: {json.dumps(v, separators=(',', ':'))}" for k, v in sorted(_answers.items()))
        gz.write(("{\n" + ",\n".join(lines) + "\n}\n").encode())


class Calls:
    """The sequence of calls of one reference object in one test (key: test module::test name#object), each stored as
    [name, inputs digest, answer]."""

    def __init__(self, key: str, real):
        self.key, self.real = key, real
        if real is not None:
            self.seq = _load()[key] = []
        else:
            if key not in _load():
                raise AssertionError(f"no recorded reference answers for {key}")
            self.it = iter(_load()[key])

    def put(self, name, inputs, value):
        self.seq.append([name, inputs, value])

    def get(self, name, inputs):
        got = next(self.it, None)
        assert got is not None and got[:2] == [name, inputs], \
            f"{self.key}: the reference was not asked this {name} call when the answers were recorded (recorded: {got and got[:2]})"
        return got[2]

    def finish(self):
        """called after the test: every recorded call must have been made"""
        if self.real is None:
            left = len(list(self.it))
            assert left == 0, f"{self.key}: {left} recorded reference calls were not made"


def recording(available) -> bool:
    """True when this session records: FPNGB_RECORD_REFERENCE is set.  Recording without the reference is an error."""
    if not RECORD:
        return False
    assert available(), "FPNGB_RECORD_REFERENCE is set but oracle/_ref is not built"
    return True


def answer_key(request, what: str) -> str:
    return f"{os.path.basename(request.node.fspath)}::{request.node.name}#{what}"


def _pixels(oracle, calls, data, desired, d):
    """the reference's decoded pixels, recomputed by the oracle's decoder and checked against the recorded digest"""
    if d is None:
        return None
    st, px, *_ = oracle.decode(data, desired)
    assert st == 0 and digest(px) == d, f"{calls.key}: the oracle's pixels differ from the reference's recorded pixels"
    return px


def _encoded(oracle, calls, png, d):
    assert digest(png) == d, f"{calls.key}: the oracle's file differs from the reference's recorded file"
    return png


class RecordedRef:
    """oracle.pyoracle.Ref: the reference encoder and decoder, lodepng and stb_image"""

    def __init__(self, calls: Calls, oracle):
        self.c, self.o, self.r = calls, oracle, calls.real

    def encode(self, img, w, h, chans, flags=0) -> bytes:
        i = inputs_digest(img, w, h, chans, flags)
        if self.r:
            png = self.r.encode(img, w, h, chans, flags)
            self.c.put("encode", i, digest(png))
            return png
        return _encoded(self.o, self.c, self.o.encode(img, w, h, chans, flags), self.c.get("encode", i))

    def get_info(self, data):
        i = inputs_digest(data)
        if self.r:
            res = self.r.get_info(data)
            self.c.put("get_info", i, list(res))
            return res
        return tuple(self.c.get("get_info", i))

    def decode(self, data, desired):
        i = inputs_digest(data, desired)
        if self.r:
            st, px, w, h, c = res = self.r.decode(data, desired)
            self.c.put("decode", i, [st, None if px is None else digest(px), w, h, c])
            return res
        st, d, w, h, c = self.c.get("decode", i)
        return st, _pixels(self.o, self.c, data, desired, d), w, h, c

    def lodepng_decode(self, data, want_chans):
        i = inputs_digest(data, want_chans)
        if self.r:
            err, px, w, h = res = self.r.lodepng_decode(data, want_chans)
            self.c.put("lodepng_decode", i, [err, None if px is None else digest(px), w, h])
            return res
        err, d, w, h = self.c.get("lodepng_decode", i)
        return err, _pixels(self.o, self.c, data, want_chans, d), w, h

    def stb_decode(self, data, want_chans):
        i = inputs_digest(data, want_chans)
        if self.r:
            comp, px, w, h = res = self.r.stb_decode(data, want_chans)
            self.c.put("stb_decode", i, [comp, None if px is None else digest(px), w, h])
            return res
        comp, d, w, h = self.c.get("stb_decode", i)
        return comp, _pixels(self.o, self.c, data, want_chans, d), w, h


class RecordedVerifiers:
    """oracle.pyoracle.Verifiers: wuffs (checksums verified) and pvpng"""

    def __init__(self, calls: Calls, oracle):
        self.c, self.o, self.r = calls, oracle, calls.real

    def wuffs_decode_rgba(self, data, w_hint, h_hint, ignore_checksums=False):
        i = inputs_digest(data, w_hint, h_hint, ignore_checksums)
        if self.r:
            rc, px, w, h = res = self.r.wuffs_decode_rgba(data, w_hint, h_hint, ignore_checksums)
            self.c.put("wuffs", i, [rc, None if px is None else digest(px), w, h])
            return res
        rc, d, w, h = self.c.get("wuffs", i)
        return rc, _pixels(self.o, self.c, data, 4, d), w, h

    def pvpng_decode(self, data, desired_chans, w_hint, h_hint):
        i = inputs_digest(data, desired_chans, w_hint, h_hint)
        if self.r:
            rc, px, w, h, c = res = self.r.pvpng_decode(data, desired_chans, w_hint, h_hint)
            self.c.put("pvpng", i, [rc, None if px is None else digest(px), w, h, c])
            return res
        rc, d, w, h, c = self.c.get("pvpng", i)
        return rc, _pixels(self.o, self.c, data, desired_chans, d), w, h, c


class RecordedTrainer:
    """oracle.pyoracle.RefTrainer: the reference built with FPNG_TRAIN_HUFFMAN_TABLES=1 (its answers are stored whole)"""

    def __init__(self, calls: Calls):
        self.c, self.r = calls, calls.real

    def counts_from_encodes(self, images, w, h, chans):
        i = inputs_digest(*images, w, h, chans)
        if self.r:
            counts = self.r.counts_from_encodes(images, w, h, chans)
            self.c.put("counts", i, [int(v) for v in counts])
            return counts
        return np.array(self.c.get("counts", i), np.uint64)

    def create_prefix(self, counts, chans):
        i = inputs_digest(np.ascontiguousarray(counts, dtype=np.uint64), chans)
        if self.r:
            prefix, bb, bs, codes, sizes = res = self.r.create_prefix(counts, chans)
            self.c.put("prefix", i, [prefix.hex(), int(bb), int(bs), [int(v) for v in codes], [int(v) for v in sizes]])
            return res
        prefix, bb, bs, codes, sizes = self.c.get("prefix", i)
        return bytes.fromhex(prefix), bb, bs, np.array(codes, np.uint32), np.array(sizes, np.uint8)


class RecordedPatched:
    """oracle.pyoracle.RefPatched: the reference encoder with a trained table patched in; the replayed files are recomputed by
    the oracle, which the calling test sets to the same table"""

    def __init__(self, calls: Calls, oracle):
        self.c, self.o, self.r = calls, oracle, calls.real

    def set_table(self, chans, prefix, bit_buf, bit_buf_size, codes, sizes) -> bool:
        i = inputs_digest(chans, bytes(prefix), bit_buf, bit_buf_size, [int(v) for v in codes], [int(v) for v in sizes])
        if self.r:
            ok = self.r.set_table(chans, prefix, bit_buf, bit_buf_size, codes, sizes)
            self.c.put("set_table", i, ok)
            return ok
        return self.c.get("set_table", i)

    def reset_table(self, chans) -> None:
        if self.r:
            self.r.reset_table(chans)

    def encode(self, img, w, h, chans, flags=0) -> bytes:
        i = inputs_digest(img, w, h, chans, flags)
        if self.r:
            png = self.r.encode(img, w, h, chans, flags)
            self.c.put("encode", i, digest(png))
            return png
        return _encoded(self.o, self.c, self.o.encode(img, w, h, chans, flags), self.c.get("encode", i))


def _harness_inputs(args, cwd: str) -> str:
    """the arguments (the run's directory written as <tmp>), the files they name and, for an @listing, the files it lists"""
    parts = []
    for a in args:
        parts.append(a.replace(cwd, "<tmp>"))
        path = os.path.join(cwd, a[1:] if a.startswith("@") else a)
        if os.path.isfile(path):
            with open(path, "rb") as f:
                data = f.read()
            parts.append(data.replace(cwd.encode(), b"<tmp>"))
            if a.startswith("@"):
                for name in data.decode().split():
                    if os.path.isfile(name):
                        with open(name, "rb") as f:
                            parts.append(f.read())
    return inputs_digest(*parts)


class RecordedHarness:
    """The reference's fpng_test program (compiled in training mode into oracle/_ref/fpng_test_train): exit status, standard
    output (with the run's temporary directory written as <tmp>) and the digest of the fpng.png it writes."""

    def __init__(self, calls: Calls):
        self.c, self.exe = calls, calls.real

    def run(self, args, cwd):
        cwd = str(cwd)
        i = _harness_inputs(args, cwd)
        if self.exe:
            r = subprocess.run([self.exe, *args], capture_output=True, text=True, cwd=cwd)
            out = os.path.join(cwd, "fpng.png")
            written = digest(open(out, "rb").read()) if os.path.exists(out) else None
            self.c.put("run", i, [r.returncode, r.stdout.replace(cwd, "<tmp>"), r.stderr[-500:], written])
            if written:
                os.remove(out)
        else:
            rc, stdout, stderr, written = self.c.get("run", i)
            r = subprocess.CompletedProcess(args, rc, stdout.replace("<tmp>", cwd), stderr)
        return r, None if written is None else Digest(written)
