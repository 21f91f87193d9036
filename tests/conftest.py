import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `pytest -m gpu`)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.pyoracle import Oracle
    return Oracle()


# The reference's answers come from tests/golden/reference_answers.json.gz (see tests/reference_answers.py): the reference is not
# part of this repository.  With FPNGB_RECORD_REFERENCE set they come from the compiled reference (oracle/_ref) and are recorded.
# After the test, every recorded call must have been made.
@pytest.fixture
def ref(request, oracle):
    """The unmodified reference encoder and decoder, lodepng and stb_image."""
    import reference_answers as ra
    from oracle.pyoracle import Ref
    real = Ref() if ra.recording(Ref.available) else None
    calls = ra.Calls(ra.answer_key(request, "ref"), real)
    yield ra.RecordedRef(calls, oracle)
    calls.finish()


@pytest.fixture
def verifiers(request, oracle):
    """wuffs (verifies IDAT CRC-32 and zlib Adler-32) and pvpng: the other two independent decoders of the reference's round-trip
    check (src/fpng_test.cpp:1403-1445, 1571-1606), compiled unmodified from the reference tree (oracle/verifiers_shim.cpp)."""
    import reference_answers as ra
    from oracle.pyoracle import Verifiers
    real = Verifiers() if ra.recording(Verifiers.available) else None
    calls = ra.Calls(ra.answer_key(request, "verifiers"), real)
    yield ra.RecordedVerifiers(calls, oracle)
    calls.finish()


@pytest.fixture
def ref_trainer(request):
    """The reference built with its FPNG_TRAIN_HUFFMAN_TABLES=1 switch: histogram accumulation and create_dynamic_block_prefix."""
    import reference_answers as ra
    from oracle.pyoracle import RefTrainer
    real = RefTrainer() if ra.recording(RefTrainer.available) else None
    calls = ra.Calls(ra.answer_key(request, "trainer"), real)
    yield ra.RecordedTrainer(calls)
    calls.finish()


@pytest.fixture
def ref_patched(request, oracle):
    """The reference encoder with its static 1-pass tables patched in memory (oracle/ref_patch_shim.cpp)."""
    import reference_answers as ra
    from oracle.pyoracle import RefPatched
    real = RefPatched() if ra.recording(RefPatched.available) else None
    calls = ra.Calls(ra.answer_key(request, "patched"), real)
    yield ra.RecordedPatched(calls, oracle)
    calls.finish()


@pytest.fixture(scope="session")
def gpu():
    import fpng_b200
    fpng_b200.fpng_init()
    return fpng_b200
