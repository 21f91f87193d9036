"""ctypes front-end for the TEST-ONLY checkers under oracle/.

* ``Oracle``  -> oracle/liboracle.so   (our C restatement, oracle/fpng_oracle.c; always buildable)
* ``Ref``     -> oracle/_ref/libfpng_ref.so (the unmodified reference + lodepng + stb_image, built from
                 /root/reference/src by oracle/Makefile when that tree exists; travels prebuilt to the GPU box)
* ``Verifiers`` -> oracle/_ref/libpng_verifiers.so (wuffs + pvpng, the other two independent decoders of the reference's
                 round-trip check, src/fpng_test.cpp:1403-1445 / 1571-1606; same build rule)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this module.
The product package (fpng_b200) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle.so")
REF_SO = os.path.join(HERE, "_ref", "libfpng_ref.so")
REF_TRAIN_SO = os.path.join(HERE, "_ref", "libfpng_ref_train.so")
REF_PATCH_SO = os.path.join(HERE, "_ref", "libfpng_ref_patch.so")
VERIFIERS_SO = os.path.join(HERE, "_ref", "libpng_verifiers.so")

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)


def build(force: bool = False) -> None:
    """Compile liboracle.so (and _ref/libfpng_ref.so when the reference sources are present)."""
    src = os.path.join(HERE, "fpng_oracle.c")
    stale = (not os.path.exists(ORACLE_SO)) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(src)
    ref_possible = os.path.exists("/root/reference/src/fpng.cpp")
    ref_stale = ref_possible and (
        (not os.path.exists(REF_SO)) or os.path.getmtime(REF_SO) < os.path.getmtime(os.path.join(HERE, "ref_shim.cpp"))
        or (not os.path.exists(REF_TRAIN_SO)) or os.path.getmtime(REF_TRAIN_SO) < os.path.getmtime(os.path.join(HERE, "ref_train_shim.cpp"))
        or (not os.path.exists(REF_PATCH_SO)) or os.path.getmtime(REF_PATCH_SO) < os.path.getmtime(os.path.join(HERE, "ref_patch_shim.cpp"))
        or (not os.path.exists(VERIFIERS_SO)) or os.path.getmtime(VERIFIERS_SO) < os.path.getmtime(os.path.join(HERE, "verifiers_shim.cpp"))
        or not os.path.exists(os.path.join(HERE, "_ref", "fpng_test_train")))
    if force or stale or ref_stale:
        subprocess.check_call(["make", "-s", "-f", os.path.join(HERE, "Makefile"), "all"], cwd=HERE)


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _as_u8(buf) -> np.ndarray:
    if isinstance(buf, np.ndarray):
        return np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
    return np.frombuffer(bytes(buf), dtype=np.uint8)


class Oracle:
    def __init__(self):
        build()
        L = C.CDLL(ORACLE_SO)
        L.oracle_init.restype = None
        L.oracle_crc32.restype = C.c_uint32
        L.oracle_crc32.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32]
        L.oracle_adler32.restype = C.c_uint32
        L.oracle_adler32.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32]
        L.oracle_max_encoded_size.restype = C.c_size_t
        L.oracle_max_encoded_size.argtypes = [C.c_uint32] * 3
        L.oracle_encode_ex.restype = C.c_size_t
        L.oracle_encode_ex.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                       C.c_size_t, C.c_void_p, C.POINTER(C.c_int)]
        L.oracle_decode.restype = C.c_int
        L.oracle_decode.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, u32p, u32p, u32p, C.c_uint32]
        L.oracle_get_info.restype = C.c_int
        L.oracle_get_info.argtypes = [C.c_void_p, C.c_uint32, u32p, u32p, u32p]
        L.oracle_static_table.restype = None
        L.oracle_static_table.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, u32p]
        L.oracle_set_static_table.restype = C.c_int
        L.oracle_set_static_table.argtypes = [C.c_uint32, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32]
        L.oracle_init()
        self.L = L

    def set_static_table(self, chans, prefix: bytes = b"", bit_buf: int = 0, bit_buf_size: int = 0) -> bool:
        """Install a trained 1-pass table (or restore the shipped one with an empty prefix)."""
        a = np.frombuffer(bytes(prefix), dtype=np.uint8) if prefix else np.zeros(1, np.uint8)
        return bool(self.L.oracle_set_static_table(chans, _ptr(a), len(prefix), bit_buf, bit_buf_size))

    def crc32(self, data, prev=0) -> int:
        a = _as_u8(data)
        return self.L.oracle_crc32(_ptr(a), a.size, prev)

    def adler32(self, data, prev=1) -> int:
        a = _as_u8(data)
        return self.L.oracle_adler32(_ptr(a), a.size, prev)

    def max_encoded_size(self, w, h, chans) -> int:
        return self.L.oracle_max_encoded_size(w, h, chans)

    def encode(self, img, w, h, chans, flags=0, want_rows=False):
        a = _as_u8(img)
        assert a.size == w * h * chans
        cap = self.max_encoded_size(w, h, chans)
        out = np.empty(cap, dtype=np.uint8)
        rows = np.zeros(h, dtype=np.uint64) if want_rows else None
        stored = C.c_int(0)
        n = self.L.oracle_encode_ex(_ptr(a), w, h, chans, flags, _ptr(out), cap,
                                    _ptr(rows) if want_rows else None, C.byref(stored))
        if n == 0:
            raise ValueError("oracle_encode rejected the arguments")
        data = out[:n].tobytes()
        if want_rows:
            return data, rows, bool(stored.value)
        return data

    def static_table(self, chans):
        sizes = np.zeros(288, np.uint8)
        codes = np.zeros(288, np.uint16)
        hb = C.c_uint32(0)
        self.L.oracle_static_table(chans, _ptr(sizes), _ptr(codes), C.byref(hb))
        return sizes, codes, hb.value

    def get_info(self, data):
        a = _as_u8(data)
        w, h, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
        st = self.L.oracle_get_info(_ptr(a), a.size, C.byref(w), C.byref(h), C.byref(c))
        return st, w.value, h.value, c.value

    def decode(self, data, desired):
        a = _as_u8(data)
        st, w, h, c = self.get_info(a)
        cap = max(1, w * h * max(desired, 1)) if st == 0 and desired in (3, 4) else 1
        out = np.empty(cap, dtype=np.uint8)
        ww, hh, cc = C.c_uint32(), C.c_uint32(), C.c_uint32()
        st = self.L.oracle_decode(_ptr(a), a.size, _ptr(out), cap, C.byref(ww), C.byref(hh), C.byref(cc), desired)
        px = out[: ww.value * hh.value * desired].copy() if st == 0 else None
        return st, px, ww.value, hh.value, cc.value


class Ref:
    """The compiled, unmodified reference (fpng v1.0.6) plus lodepng and stb_image verifiers."""

    @staticmethod
    def available() -> bool:
        try:
            build()
        except Exception:
            pass
        return os.path.exists(REF_SO)

    def __init__(self):
        if not Ref.available():
            raise RuntimeError("oracle/_ref/libfpng_ref.so is not built (reference sources absent?)")
        L = C.CDLL(REF_SO)
        L.ref_init.restype = None
        L.ref_cpu_supports_sse41.restype = C.c_int
        L.ref_crc32.restype = C.c_uint32
        L.ref_crc32.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32]
        L.ref_adler32.restype = C.c_uint32
        L.ref_adler32.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32]
        L.ref_encode.restype = C.c_size_t
        L.ref_encode.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t]
        L.ref_encode_discard.restype = C.c_size_t
        L.ref_encode_discard.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int]
        L.ref_decode_discard.restype = C.c_int
        L.ref_decode_discard.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]
        L.ref_get_info.restype = C.c_int
        L.ref_get_info.argtypes = [C.c_void_p, C.c_uint32, u32p, u32p, u32p]
        L.ref_decode.restype = C.c_int
        L.ref_decode.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, u32p, u32p, u32p, C.c_uint32]
        L.ref_lodepng_decode.restype = C.c_uint
        L.ref_lodepng_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, u32p, u32p, C.c_uint32]
        L.ref_stb_decode.restype = C.c_int
        L.ref_stb_decode.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, u32p, u32p, C.c_int]
        L.ref_init()
        self.L = L

    def sse41(self) -> bool:
        return bool(self.L.ref_cpu_supports_sse41())

    def crc32(self, data, prev=0):
        a = _as_u8(data)
        return self.L.ref_crc32(_ptr(a), a.size, prev)

    def adler32(self, data, prev=1):
        a = _as_u8(data)
        return self.L.ref_adler32(_ptr(a), a.size, prev)

    def encode(self, img, w, h, chans, flags=0) -> bytes:
        a = _as_u8(img)
        assert a.size == w * h * chans
        cap = 58 + 6 + (w * chans + 1) * h + 5 * (((w * chans + 1) * h + 65534) // 65535) + 16 + 64
        out = np.empty(cap, dtype=np.uint8)
        n = self.L.ref_encode(_ptr(a), w, h, chans, flags, _ptr(out), cap)
        if n == 0 or n > cap:
            raise ValueError("reference encoder failed")
        return out[:n].tobytes()

    def encode_discard(self, img, w, h, chans, flags=0, reps=1) -> int:
        a = _as_u8(img)
        return self.L.ref_encode_discard(_ptr(a), w, h, chans, flags, reps)

    def decode_discard(self, data, desired, reps=1) -> int:
        a = _as_u8(data)
        return self.L.ref_decode_discard(_ptr(a), a.size, desired, reps)

    def get_info(self, data):
        a = _as_u8(data)
        w, h, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
        st = self.L.ref_get_info(_ptr(a), a.size, C.byref(w), C.byref(h), C.byref(c))
        return st, w.value, h.value, c.value

    def decode(self, data, desired):
        a = _as_u8(data)
        st, w, h, c = self.get_info(a)
        cap = max(1, w * h * 4)
        out = np.empty(cap, dtype=np.uint8)
        ww, hh, cc = C.c_uint32(), C.c_uint32(), C.c_uint32()
        st = self.L.ref_decode(_ptr(a), a.size, _ptr(out), cap, C.byref(ww), C.byref(hh), C.byref(cc), desired)
        px = out[: ww.value * hh.value * desired].copy() if st == 0 else None
        return st, px, ww.value, hh.value, cc.value

    def lodepng_decode(self, data, want_chans):
        a = _as_u8(data)
        st, w, h, c = self.get_info(a)
        if w == 0 or h == 0:   # not parsable by fpng's walker: let lodepng find dimensions with a big buffer
            w, h = 8192, 8192
        out = np.empty(w * h * want_chans, dtype=np.uint8)
        ww, hh = C.c_uint32(), C.c_uint32()
        err = self.L.ref_lodepng_decode(_ptr(a), a.size, _ptr(out), out.size, C.byref(ww), C.byref(hh), want_chans)
        px = out[: ww.value * hh.value * want_chans].copy() if err == 0 else None
        return err, px, ww.value, hh.value

    def stb_decode(self, data, want_chans):
        a = _as_u8(data)
        st, w, h, c = self.get_info(a)
        out = np.empty(max(1, w * h * want_chans), dtype=np.uint8)
        ww, hh = C.c_uint32(), C.c_uint32()
        comp = self.L.ref_stb_decode(_ptr(a), a.size, _ptr(out), out.size, C.byref(ww), C.byref(hh), want_chans)
        px = out[: ww.value * hh.value * want_chans].copy() if comp else None
        return comp, px, ww.value, hh.value


class Verifiers:
    """wuffs (checksums verified) and pvpng, compiled unmodified from the reference tree (oracle/verifiers_shim.cpp)."""

    @staticmethod
    def available() -> bool:
        try:
            build()
        except Exception:
            pass
        return os.path.exists(VERIFIERS_SO)

    def __init__(self):
        if not Verifiers.available():
            raise RuntimeError("oracle/_ref/libpng_verifiers.so is not built (reference sources absent?)")
        L = C.CDLL(VERIFIERS_SO)
        L.ver_wuffs_decode_rgba.restype = C.c_int
        L.ver_wuffs_decode_rgba.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t, u32p, u32p]
        L.ver_pvpng_decode.restype = C.c_int
        L.ver_pvpng_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p, C.c_size_t, u32p, u32p, u32p]
        self.L = L

    def wuffs_decode_rgba(self, data, w_hint: int, h_hint: int, ignore_checksums: bool = False):
        """-> (rc, pixels[h*w*4] or None, w, h); rc 0 = decoded AND (unless ignored) IDAT CRC-32 / zlib Adler-32 correct"""
        a = _as_u8(data)
        out = np.empty(max(1, w_hint * h_hint * 4), dtype=np.uint8)
        ww, hh = C.c_uint32(), C.c_uint32()
        rc = self.L.ver_wuffs_decode_rgba(_ptr(a), a.size, int(ignore_checksums), _ptr(out), out.size, C.byref(ww), C.byref(hh))
        return rc, (out[: ww.value * hh.value * 4].copy() if rc == 0 else None), ww.value, hh.value

    def pvpng_decode(self, data, desired_chans: int, w_hint: int, h_hint: int):
        """-> (rc, pixels[h*w*desired] or None, w, h, channels in file)"""
        a = _as_u8(data)
        out = np.empty(max(1, w_hint * h_hint * desired_chans), dtype=np.uint8)
        ww, hh, cc = C.c_uint32(), C.c_uint32(), C.c_uint32()
        rc = self.L.ver_pvpng_decode(_ptr(a), a.size, desired_chans, _ptr(out), out.size, C.byref(ww), C.byref(hh), C.byref(cc))
        return rc, (out[: ww.value * hh.value * desired_chans].copy() if rc == 0 else None), ww.value, hh.value, cc.value


class RefTrainer:
    """The reference built with FPNG_TRAIN_HUFFMAN_TABLES=1: g_huff_counts accumulation + create_dynamic_block_prefix."""

    @staticmethod
    def available() -> bool:
        try:
            build()
        except Exception:
            pass
        return os.path.exists(REF_TRAIN_SO)

    def __init__(self):
        if not RefTrainer.available():
            raise RuntimeError("oracle/_ref/libfpng_ref_train.so is not built")
        L = C.CDLL(REF_TRAIN_SO)
        L.reft_encode.restype = C.c_size_t
        L.reft_encode.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.reft_get_counts.argtypes = [C.c_void_p]
        L.reft_create_prefix.restype = C.c_int
        L.reft_create_prefix.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_uint64),
                                         C.POINTER(C.c_int), C.c_void_p, C.c_void_p]
        L.reft_init()
        self.L = L

    def counts_from_encodes(self, images, w, h, chans):
        self.L.reft_reset_counts()
        for im in images:
            a = _as_u8(im)
            assert self.L.reft_encode(_ptr(a), w, h, chans, 1) > 0
        out = np.zeros(288, np.uint64)
        self.L.reft_get_counts(_ptr(out))
        return out

    def create_prefix(self, counts, chans):
        counts = np.ascontiguousarray(counts, dtype=np.uint64)
        prefix = np.zeros(4096, np.uint8); n = C.c_size_t(); bb = C.c_uint64(); bs = C.c_int()
        codes = np.zeros(288, np.uint32); sizes = np.zeros(288, np.uint8)
        ok = self.L.reft_create_prefix(_ptr(counts), chans, _ptr(prefix), prefix.size, C.byref(n), C.byref(bb), C.byref(bs), _ptr(codes), _ptr(sizes))
        assert ok
        return prefix[: n.value].tobytes(), bb.value, bs.value, codes, sizes


class RefPatched:
    """The reference encoder with its static 1-pass tables patchable in memory (oracle/ref_patch_shim.cpp): every line of
    the encoder is the reference's, only the table contents change.  Prefix length must equal the reference's own
    compile-time table size (62 bytes RGB / 61 bytes RGBA)."""

    @staticmethod
    def available() -> bool:
        try:
            build()
        except Exception:
            pass
        return os.path.exists(REF_PATCH_SO)

    def __init__(self):
        if not RefPatched.available():
            raise RuntimeError("oracle/_ref/libfpng_ref_patch.so is not built")
        L = C.CDLL(REF_PATCH_SO)
        L.refp_table_len.restype = C.c_uint32
        L.refp_table_len.argtypes = [C.c_uint32]
        L.refp_set_table.restype = C.c_int
        L.refp_set_table.argtypes = [C.c_uint32, C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
        L.refp_reset_table.argtypes = [C.c_uint32]
        L.refp_encode.restype = C.c_size_t
        L.refp_encode.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t]
        L.refp_decode.restype = C.c_int
        L.refp_decode.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, u32p, u32p, u32p, C.c_uint32]
        L.refp_init()
        self.L = L

    def table_len(self, chans) -> int:
        return self.L.refp_table_len(chans)

    def set_table(self, chans, prefix: bytes, bit_buf: int, bit_buf_size: int, codes, sizes) -> bool:
        pre = np.frombuffer(bytes(prefix), dtype=np.uint8).copy()
        codes = np.ascontiguousarray(codes, dtype=np.uint32)
        sizes = np.ascontiguousarray(sizes, dtype=np.uint8)
        return bool(self.L.refp_set_table(chans, _ptr(pre), pre.size, bit_buf, bit_buf_size, _ptr(codes), _ptr(sizes)))

    def reset_table(self, chans) -> None:
        self.L.refp_reset_table(chans)

    def encode(self, img, w, h, chans, flags=0) -> bytes:
        a = _as_u8(img).copy()
        cap = 58 + 6 + (w * chans + 1) * h + 5 * (((w * chans + 1) * h + 65534) // 65535) + 16 + 64
        out = np.empty(cap, dtype=np.uint8)
        n = self.L.refp_encode(_ptr(a), w, h, chans, flags, _ptr(out), cap)
        if n == 0 or n > cap:
            raise ValueError("patched reference encoder failed")
        return out[:n].tobytes()
