"""Checksums of row ranges of an index image, on the host (host/image.py): a section's checksum counts word positions
from the image's row 0, so the checksums of slices taken at their offsets add up, mod 2^64, to the section's."""
import numpy as np


def _image():
    import importlib
    import bbq_b200  # noqa: F401  (registers the package under its importable name)
    return importlib.import_module("better_binary_quantization_b200.host.image")


def test_offset_slices_sum_to_the_whole_section():
    img = _image()
    rng = np.random.default_rng(5)
    for stride in (4, 8, 16, 96):                               # componentSum, f64 columns, code rows of 100 and 768 dims
        rows = 1001
        raw = rng.integers(0, 2**32, rows * stride // 4, dtype=np.uint64).astype("<u4").tobytes()
        whole = img.section_checksum(raw)
        for bounds in ([0, rows], [0, 1, rows], [0, 7, 7, 500, 999, rows]):
            total = 0
            for r0, r1 in zip(bounds[:-1], bounds[1:]):
                total += img.section_checksum(raw[r0 * stride:r1 * stride], first_word=r0 * stride // 4)
            assert total & 0xFFFFFFFFFFFFFFFF == whole, (stride, bounds)
        # a slice checksummed from the wrong position does not fit
        assert img.section_checksum(raw[stride:]) + img.section_checksum(raw[:stride]) != whole


def test_first_word_known_answer():
    img = _image()
    import struct
    # one zero word at position p: splitmix64(p << 32); position 0 is the known answer of test_index_image.py
    assert img.section_checksum(struct.pack("<I", 0), first_word=0) == 0xE220A8397B1DCDAF
    two = struct.pack("<II", 0, 0)
    assert img.section_checksum(two) == (img.section_checksum(two[:4]) + img.section_checksum(two[4:], first_word=1)) % 2**64
