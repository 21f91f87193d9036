"""Tests against the REAL reference harness (fpng_test compiled from the reference sources, test-only, into oracle/_ref/; its
recorded output, tests/reference_answers.py, where the reference is absent).

1. tools/train_tables.py (the `fpng_test -t` counterpart) against the REAL harness: the unmodified reference's fpng_test is compiled
with its own FPNG_TRAIN_HUFFMAN_TABLES=1 switch (into oracle/_ref/, test-only) and run on a listing of PNG files; the driver -- with
the reference trainer (oracle/_ref/libfpng_ref_train.so) standing in for the GPU backend, since this test has no device -- must print
the same text: per-file lines (dimensions, alpha detection src/fpng_test.cpp:808-821), totals, and both C tables character for
character (src/fpng_test.cpp:893-961).  The GPU backend's two calls (histogram accumulation, prefix builder) are pinned to the same
reference trainer by tests/test_training_gpu.py.

2. BASELINE config 1 through the harness's own plumbing (see test_config1_through_the_real_harness_plumbing)."""
import io
import os
import sys

import numpy as np
import pytest

import imagegen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "oracle", "_ref", "fpng_test_train")


@pytest.fixture
def harness(request):
    """fpng_test built in training mode (same encoder output) by oracle/Makefile, as recorded (tests/reference_answers.py)"""
    import reference_answers as ra
    real = HARNESS if ra.recording(lambda: os.path.exists(HARNESS)) else None
    calls = ra.Calls(ra.answer_key(request, "harness"), real)
    yield ra.RecordedHarness(calls)
    calls.finish()


class ReferenceTrainerBackend:
    """stands in for tools/train_tables.py GpuBackend (same three calls) on a box without a device"""

    def __init__(self, trainer, ref):
        self.t, self.ref = trainer, ref

    def accumulate(self, img, counts):
        h, w, c = img.shape
        counts += self.t.counts_from_encodes([img], w, h, c)

    def create_prefix(self, counts, chans):
        return self.t.create_prefix(counts, chans)

    def sanity(self, img):
        h, w, c = img.shape
        st, px, *_ = self.ref.decode(self.ref.encode(img, w, h, c, 1), c)
        return st == 0 and np.array_equal(px, img.reshape(-1))


def _write_pngs(tmp, oracle):
    names = []
    cases = [("g1", 96, 40, 3), ("g1", 64, 64, 4), ("g0", 200, 30, 4), ("runs", 150, 20, 3), ("g2", 31, 17, 3), ("mut", 120, 33, 4),
             ("g1", 50, 50, 4)]
    for i, (kind, w, h, c) in enumerate(cases):
        img = np.asarray(imagegen.make(kind, w, h, c, i)).reshape(h, w, c).copy()
        if i == 6:
            img[:, :, 3] = 255                                  # an RGBA file whose alpha is all opaque trains the 24bpp table (Q8)
        p = os.path.join(tmp, f"img{i}.png")
        with open(p, "wb") as f:
            f.write(oracle.encode(img, w, h, c, 0))
        names.append(p)
    bad = os.path.join(tmp, "broken.png")
    with open(bad, "wb") as f:
        f.write(b"not a png at all")
    names.insert(3, bad)                                        # skipped with a warning, counted as failed
    listing = os.path.join(tmp, "list.txt")
    with open(listing, "w") as f:
        f.write("\n".join(names) + "\n\n")
    return listing


def test_training_driver_prints_what_the_real_harness_prints(tmp_path, oracle, harness, ref_trainer, ref):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import train_tables
    listing = _write_pngs(str(tmp_path), oracle)
    real, _ = harness.run(["-t", "@" + listing], cwd=tmp_path)
    assert real.returncode == 0, real.stderr
    # the harness prints a banner / SSE line first; compare from the listing line on
    real_lines = real.stdout.splitlines()
    start = next(i for i, l in enumerate(real_lines) if l.startswith("Successfully read"))
    buf = io.StringIO()
    files = train_tables.load_listing("@" + listing)
    assert len(files) == 8
    tables = train_tables.train(files, ReferenceTrainerBackend(ref_trainer, ref), out=buf)
    mine = [real_lines[start]] + buf.getvalue().splitlines()
    assert mine == real_lines[start:], "\n".join(f"{a!r}\n{b!r}" for a, b in zip(mine, real_lines[start:]) if a != b)
    assert "Total alpha files: 3" in mine and "Total opaque files: 4" in mine and "Total failed loading: 1" in mine
    assert tables[3] is not None and tables[4] is not None and len(tables[3][0]) > 40


@pytest.mark.parametrize("opts,flags", [((), 0), (("-s",), 1), (("-u",), 2)])
def test_config1_through_the_real_harness_plumbing(tmp_path, oracle, harness, opts, flags):
    """BASELINE config 1 ("single 512x512 RGBA synthetic gradient, 1-pass encode ... (fpng_test plumbing)") through the REAL harness:
    the G0 image (alpha = green ramp, so fpng_test's alpha auto-detect keeps it 32bpp, src/fpng_test.cpp:1156-1166) is written as a
    general PNG, `fpng_test [-s|-u]` loads it with lodepng, encodes, verifies with its five decoders and writes fpng.png
    (src/fpng_test.cpp:1216) -- which must be byte for byte what the oracle (and therefore the GPU encoder, tests/test_encode_gpu.py)
    produces for the same pixels and flags.  The harness binary is the training-mode build used above (same encoder output)."""
    from PIL import Image
    import bench
    wl = bench.WORKLOADS["c1"]
    w, h, c = wl["w"], wl["h"], wl["chans"]
    img = bench.workload_image(wl, "g0", 0)
    assert img.shape == (h, w, c) and (img[:, :, 3] < 255).any()
    src = tmp_path / "c1_g0.png"
    Image.fromarray(img, "RGBA").save(src)
    r, out = harness.run([*opts, str(src)], cwd=tmp_path)        # fpng.png is written without -c
    assert r.returncode == 0, r.stdout[-500:] + r.stderr[-500:]
    assert "Has Alpha: 1" in r.stdout
    assert out == oracle.encode(img, w, h, c, flags)
    r, _ = harness.run(["-c", *opts, str(src)], cwd=tmp_path)
    assert r.returncode == 0, r.stdout[-500:] + r.stderr[-500:]
    # CSV row: file, w, h, chans, then {enc s, MB, dec s, enc MP/s, dec MP/s} for qoi, fpng, lodepng, stbi, and pvpng's two
    row = [t.strip() for t in r.stdout.strip().splitlines()[-1].split(",")]
    assert row[1:4] == ["512", "512", "4"] and len(row) == 4 + 4 * 5 + 2
    assert abs(float(row[10]) - len(out) / (1024.0 * 1024.0)) < 1e-5 and float(row[12]) > 0 and float(row[13]) > 0
