"""Trained 1-pass tables on the GPU: byte parity of fpngb_set_static_table() + 1-pass encode with the reference encoder
running the same table (patched in memory, oracle/ref_patch_shim.cpp), with the oracle, and with the committed digests.
Under the RGBA fixture table the "one-pixel match vs four literals" check (src/fpng.cpp:1520-1528) fires 186 times."""
import numpy as np
import pytest

import imagegen
from common import sha
from test_trained_tables_cpu import load_tables

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("chans", [3, 4])
def test_trained_table_byte_parity(gpu, oracle, ref, ref_patched, chans):
    import torch
    t = load_tables()[str(chans)]
    prefix = bytes.fromhex(t["prefix"])
    sizes = np.array(t["sizes"], np.uint8)
    rp = ref_patched
    assert rp.set_table(chans, prefix, t["bit_buf"], t["bit_buf_size"], t["codes"], t["sizes"])
    assert oracle.set_static_table(chans, prefix, t["bit_buf"], t["bit_buf_size"])
    try:
        gpu.set_static_table(chans, prefix, t["bit_buf"], t["bit_buf_size"])
        for (name, w, h, img), vec in zip(imagegen.trained_table_images(chans, sizes), t["vectors"]):
            ok, png = gpu.fpng_encode_image_to_memory(img, w, h, chans, 0)
            assert ok
            assert sha(png) == vec["sha256"], (name, len(png), vec["size"])
            assert png == oracle.encode(img, w, h, chans, 0), name
            assert png == rp.encode(img, w, h, chans, 0), name
            st, px, *_ = ref.decode(png, chans)                      # the unmodified reference decoder reads the table from the stream
            assert st == 0 and np.array_equal(px, img.reshape(-1))
            st, px, *_ = gpu.fpng_decode_memory(png, chans)
            assert st == 0 and np.array_equal(px, img.reshape(-1))
        # the batch entry point (device-resident, several images, 16-byte aligned rows) takes the same table
        w, h = 64, 24
        imgs = [imagegen.short_runs(w, h, chans, 7 + i, [int(v) for v in np.argsort(sizes[:256], kind="stable")[:4]]) for i in range(5)]
        dev = torch.from_numpy(np.stack(imgs)).cuda()
        out, szs = gpu.encode_batch_device(dev, 0)
        torch.cuda.synchronize()
        out = out.cpu().numpy(); szs = szs.cpu().numpy().astype(np.uint32)
        for i, im in enumerate(imgs):
            assert out[i, : szs[i]].tobytes() == oracle.encode(im, w, h, chans, 0), i
        # 2-pass and stored modes ignore the static table
        im = imgs[0]
        assert gpu.fpng_encode_image_to_memory(im, w, h, chans, 1)[1] == ref.encode(im, w, h, chans, 1)
        assert gpu.fpng_encode_image_to_memory(im, w, h, chans, 2)[1] == ref.encode(im, w, h, chans, 2)
    finally:
        gpu.set_static_table(chans)
        oracle.set_static_table(chans)
        rp.reset_table(chans)
    im = imagegen.make("g1", 64, 8, chans, 0)
    assert gpu.fpng_encode_image_to_memory(im, 64, 8, chans, 0)[1] == ref.encode(im, 64, 8, chans, 0)


def test_set_static_table_rejects_undecodable_tables(gpu):
    """ADVICE r1: literal/length sizes above 12 or a distance table other than the trainer's must be refused."""
    t = load_tables()["4"]
    prefix = bytearray(bytes.fromhex(t["prefix"]))
    from fpng_b200._lib import FpngB200Error
    with pytest.raises(FpngB200Error):
        gpu.set_static_table(4, bytes(prefix[:20]), 0, 0)             # truncated header
    gpu.set_static_table(4)
