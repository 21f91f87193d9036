"""CPU tests: the oracle (oracle/fpng_oracle.c) against the reference's known answers, the committed golden vectors
(tests/golden/reference_vectors.json, produced by the unmodified reference) and, when oracle/_ref is built, the
reference itself on the reference's fuzz families (src/fpng_test.cpp:381-682)."""
import json
import os

import numpy as np

import imagegen
from common import golden_vectors, sha


def test_checksum_known_answers(oracle):
    # SURVEY.md section 8c item 5
    assert oracle.crc32(b"123456789") == 0xCBF43926
    assert oracle.adler32(b"Wikipedia") == 0x11E60398
    # incremental chaining (src/fpng.h:27,31)
    d = bytes(range(256)) * 41
    assert oracle.crc32(d[100:], oracle.crc32(d[:100])) == oracle.crc32(d)
    assert oracle.adler32(d[100:], oracle.adler32(d[:100])) == oracle.adler32(d)


def test_oracle_matches_golden_vectors(oracle):
    vecs = golden_vectors()
    assert len(vecs) > 600
    for v in vecs:
        img = imagegen.make(v["kind"], v["w"], v["h"], v["chans"], v["index"])
        assert sha(img.tobytes()) == v["pixels_sha256"], "generator drifted"
        png = oracle.encode(img, v["w"], v["h"], v["chans"], v["flags"])
        assert len(png) == v["size"] and sha(png) == v["png_sha256"], v
        if "png_hex" in v:
            assert png.hex() == v["png_hex"]
        st, px, w, h, c = oracle.decode(png, v["chans"])
        assert st == 0 and (w, h, c) == (v["w"], v["h"], v["chans"]) and sha(px) == v["pixels_sha256"]


def test_oracle_channel_conversion(oracle):
    # 24->32: alpha 0xFF; 32->24: alpha dropped (src/fpng_test.cpp:1276-1327)
    for c in (3, 4):
        img = imagegen.make("g1", 61, 7, c, 3)
        png = oracle.encode(img, 61, 7, c, 0)
        d = 7 - c
        st, px, w, h, cc = oracle.decode(png, d)
        assert st == 0 and cc == c
        px = px.reshape(7, 61, d)
        assert np.array_equal(px[..., :3], img[..., :3])
        if d == 4:
            assert (px[..., 3] == 255).all()


def test_oracle_decode_rejects(oracle):
    img = imagegen.make("g1", 40, 6, 3, 1)
    png = bytearray(oracle.encode(img, 40, 6, 3, 0))
    assert oracle.decode(bytes(png), 5)[0] == 2                     # FPNG_DECODE_INVALID_ARG
    bad = bytearray(png); bad[0] = 0
    assert oracle.decode(bytes(bad), 3)[0] == 3                     # NOT_PNG
    bad = bytearray(png); bad[17] ^= 1                              # IHDR width -> header CRC mismatch
    assert oracle.decode(bytes(bad), 3)[0] == 4
    bad = bytearray(png); bad[41] ^= 0xFF                           # fdEC signature byte -> its CRC fails first
    assert oracle.decode(bytes(bad), 3)[0] == 4
    bad = bytearray(png); bad[70] ^= 0x55                           # corrupt the Huffman header / tokens
    assert oracle.decode(bytes(bad), 3)[0] in (1,)                  # NOT_FPNG


def _ref_cases():
    rs = np.random.RandomState(99)
    cases = []
    for trial in range(120):
        w = int(rs.randint(1, 300)); h = int(rs.randint(1, 40)); c = int(rs.choice([3, 4]))
        kind = ["g0", "g1", "g2", "runs", "mut", "zero"][trial % 6]
        if trial % 7 == 0:
            w = int(rs.randint(1, 30)); h = int(rs.randint(1, 4))
        cases.append((kind, w, h, c, trial))
    return cases


def test_oracle_byte_exact_vs_reference(oracle, ref):
    for (kind, w, h, c, idx) in _ref_cases():
        img = imagegen.make(kind, w, h, c, idx)
        for flags in (0, 1, 2):
            a = oracle.encode(img, w, h, c, flags)
            b = ref.encode(img, w, h, c, flags)
            assert a == b, (kind, w, h, c, flags)
            for d in (3, 4):
                sa, pa, *_ = oracle.decode(b, d)
                sb, pb, *_ = ref.decode(b, d)
                assert sa == sb == 0 and np.array_equal(pa, pb)
            err, px, ww, hh = ref.lodepng_decode(a, c)
            assert err == 0 and np.array_equal(px, img.reshape(-1))
            comp, px, ww, hh = ref.stb_decode(a, c)
            assert comp == c and np.array_equal(px, img.reshape(-1))


def test_oracle_decode_status_vs_reference_on_corruption(oracle, ref):
    rs = np.random.RandomState(5)
    img = imagegen.make("g1", 97, 13, 4, 2)
    png = oracle.encode(img, 97, 13, 4, 0)
    same = 0
    for t in range(300):
        bad = bytearray(png)
        pos = int(rs.randint(0, len(bad)))
        bad[pos] ^= 1 << int(rs.randint(0, 8))
        a = oracle.decode(bytes(bad), 4); b = ref.decode(bytes(bad), 4)
        assert a[0] == b[0], (pos, a[0], b[0])
        if a[0] == 0:
            assert np.array_equal(a[1], b[1])
        same += 1
    assert same == 300


def test_static_tables_match_reference_source(oracle):
    """The code tables derived from the header bytes equal the tables the reference stores (src/fpng.cpp:536-562), as read from
    its source by tests/golden/make_static_tables.py."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "static_tables.json")) as f:
        tables = json.load(f)
    for chans in (3, 4):
        pairs = list(zip(tables[str(chans)]["sizes"], tables[str(chans)]["codes"]))
        assert len(pairs) == 288
        sizes, codes, hdr_bits = oracle.static_table(chans)
        for i, (s, c) in enumerate(pairs):
            assert sizes[i] == int(s) and (int(s) == 0 or codes[i] == int(c)), (chans, i)


def test_oracle_decode_vs_reference_on_stream_mutations(oracle, ref):
    """The decoder fuzz of the reference (`fpng_test -f` under zzuf, README.md:185-189) as a seeded CPU test: byte overwrites, bit flips,
    short random splices, byte swaps and block-header damage inside the IDAT payload (its CRC is not checked by the decoder, fpng.cpp
    F9), 1-pass / 2-pass / stored files, both desired channel counts -- status AND pixels of the oracle must equal the unmodified
    reference's.  About a quarter of the mutants still decode (to different pixels): the comparison is not just 'both reject'."""
    import imagegen
    rs = np.random.RandomState(77)
    n = ok = 0
    for kind, w, h, c, fl in [("g1", 97, 31, 4, 0), ("g1", 160, 24, 3, 0), ("g0", 256, 40, 4, 0), ("runs", 300, 17, 3, 0), ("g1", 128, 32, 3, 1),
                               ("runs", 301, 9, 4, 1), ("g2", 40, 9, 3, 0), ("mut", 120, 33, 4, 0), ("g0", 333, 20, 3, 1), ("g1", 40, 12, 4, 2)]:
        png = oracle.encode(imagegen.make(kind, w, h, c, 5), w, h, c, fl)
        idat, end = png.index(b"IDAT") + 4, len(png) - 16
        for trial in range(250):
            bad = bytearray(png)
            m = rs.randint(0, 5)
            if m == 0:
                for _ in range(rs.randint(1, 4)):
                    bad[rs.randint(idat, end)] = rs.randint(0, 256)
            elif m == 1:
                bad[rs.randint(idat, end)] ^= 1 << rs.randint(0, 8)
            elif m == 2:
                p, L = rs.randint(idat, end - 8), rs.randint(1, 8)
                bad[p:p + L] = bytes(rs.randint(0, 256, L, dtype=np.uint8))
            elif m == 3:
                a, b = rs.randint(idat, end), rs.randint(idat, end)
                bad[a], bad[b] = bad[b], bad[a]
            else:
                bad[rs.randint(idat, min(idat + 70, end))] = rs.randint(0, 256)
            bad = bytes(bad)
            for d in (3, 4):
                a, b = oracle.decode(bad, d), ref.decode(bad, d)
                assert a[0] == b[0], (kind, w, h, c, fl, trial, m, d, a[0], b[0])
                if a[0] == 0:
                    assert np.array_equal(a[1], b[1]), (kind, w, h, c, fl, trial, m, d)
                    ok += 1
                n += 1
    assert n == 5000 and ok > 500
