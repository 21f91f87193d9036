"""GPU tests of the static-table training path (SURVEY section 8f rank 3): histogram accumulation and
create_dynamic_block_prefix must equal the reference built with its own FPNG_TRAIN_HUFFMAN_TABLES=1 switch; a trained
table installed for 1-pass encoding yields ordinary fpng files (reference decoder accepts them) that are smaller on the
training workload; restoring the built-in table restores byte parity with the reference."""
import numpy as np
import pytest

import imagegen

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("workload", ["mixed", "noisy"])
@pytest.mark.parametrize("chans", [3, 4])
def test_training_matches_reference(gpu, ref, ref_trainer, chans, workload):
    import torch
    w, h, n = 256, 96, 6
    kinds = ["g1", "g0", "runs"] if workload == "mixed" else ["g1"]
    imgs = [imagegen.make(kinds[i % len(kinds)], w, h, chans, i) for i in range(n)]
    dev = torch.from_numpy(np.stack(imgs)).cuda()
    counts = gpu.train_accumulate_device(dev)
    ref_counts = ref_trainer.counts_from_encodes(imgs, w, h, chans)
    assert np.array_equal(counts, ref_counts)
    got = gpu.create_dynamic_block_prefix(counts, chans)
    exp = ref_trainer.create_prefix(ref_counts, chans)
    assert got[0] == exp[0] and got[1] == exp[1] and got[2] == exp[2]
    assert np.array_equal(got[4], exp[4])                       # code sizes
    used = exp[4] != 0
    assert np.array_equal(got[3][used], exp[3][used])           # codes of every used symbol
    # install, encode 1-pass, verify with the reference decoder, compare sizes, restore
    default_sizes = [len(gpu.fpng_encode_image_to_memory(im, w, h, chans, 0)[1]) for im in imgs]
    try:
        gpu.set_static_table(chans, got[0], got[1], got[2])
        trained_sizes = []
        for im in imgs:
            ok, png = gpu.fpng_encode_image_to_memory(im, w, h, chans, 0)
            assert ok
            st, px, *_ = ref.decode(png, chans)
            assert st == 0 and np.array_equal(px, im.reshape(-1))
            err, px2, *_ = ref.lodepng_decode(png, chans)
            assert err == 0 and np.array_equal(px2, im.reshape(-1))
            st, px3, *_ = gpu.fpng_decode_memory(png, chans)
            assert st == 0 and np.array_equal(px3, im.reshape(-1))
            trained_sizes.append(len(png))
        if workload == "noisy":      # a table trained on one kind of content beats the generic table on that content
            assert sum(trained_sizes) < sum(default_sizes)
    finally:
        gpu.set_static_table(chans)
    for im in imgs[:2]:
        assert gpu.fpng_encode_image_to_memory(im, w, h, chans, 0)[1] == ref.encode(im, w, h, chans, 0)
