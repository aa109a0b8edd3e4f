"""The oracle's constant data against the reference's, as stored in tests/golden/reference_constants.json (CPU only):
the 9 + 9 quantization table families (src/quantization.rs:62-183), the four K.3 Huffman tables (src/huffman.rs:14-64)
and ZIGZAG (src/writer.rs:64-68). tests/golden/make_golden.py extracts the file from the reference's source text."""
import json
import os

import numpy as np

from oracle import oracle as orc

import t81_decoder as t81
from test_stream_exact import ZIGZAG

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_constants.json")


def _ref():
    return json.load(open(GOLD))


def test_quantization_table_families():
    ref = _ref()
    luma, chroma = ref["quantization_luma"], ref["quantization_chroma"]
    assert len(luma) == 9 and len(chroma) == 9
    for k in range(9):
        for is_luma, fam in ((True, luma), (False, chroma)):
            assert len(fam[k]) == 64
            tab, _, _ = orc.quant_table(k, 50, is_luma)  # quality 50 = scale 100: the family's own values
            assert tab == [min(255, max(1, v)) << 3 for v in fam[k]]


def test_default_huffman_tables_and_zigzag():
    ref = _ref()
    h = ref["huffman"]
    want = {(0, 0): h["luma_dc"], (1, 0): h["luma_ac"], (0, 1): h["chroma_dc"], (1, 1): h["chroma_ac"]}
    d = t81.decode(orc.encode(np.zeros((8, 8, 3), np.uint8), 8, 8, orc.RGB, quality=90))
    assert len(d.dht) == 4
    for tc, th, counts, values in d.dht:
        assert (list(counts), list(values)) == (want[(tc, th)]["counts"], want[(tc, th)]["values"])
    assert ref["zigzag"] == ZIGZAG
