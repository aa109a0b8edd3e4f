"""Regenerates the fixtures in this directory. Run in the build container only (`/root/reference` does not
exist on the GPU box):  python tests/golden/make_golden.py

* rgb_to_ycbcr_kat.json, fdct_kat.json: the literal known-answer vectors of the reference's own unit tests,
  read out of its sources (test_rgb_to_ycbcr, /root/reference/src/image_buffer.rs:324-421; test_fdct_libjpeg,
  /root/reference/src/fdct.rs:249-300).
* reference_constants.json: the reference's constant data, read out of its sources: the 9 + 9 quantization table
  families (src/quantization.rs), the four K.3 Huffman tables (src/huffman.rs) and ZIGZAG (src/writer.rs).
* oracle_jpegs.json: SHA-256 and length of the oracle's file bytes for a fixed matrix of configurations over
  deterministic images. It guards the oracle against regressions (tests/test_oracle.py) and gives the GPU
  tests a committed target that does not depend on the oracle being built (tests/test_gpu_parity.py).
"""
import hashlib
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

REF = "/root/reference/src"


def golden_matrix():
    """(name, image maker name, args, color, cfg): shared with the tests through this module."""
    m = []
    for color, maker, size in (("rgb", "ref_img_rgb", (258, 128)), ("rgba", "ref_img_rgba", (258, 128)),
                               ("luma", "ref_img_gray", (258, 128)), ("cmyk", "ref_img_cmyk", (258, 192)),
                               ("cmyk_as_ycck", "ref_img_cmyk", (258, 192))):
        for q in (100, 80, 30):
            m.append((f"{color}_q{q}", maker, size, color, {"quality": q}))
        m.append((f"{color}_prog", maker, size, color, {"quality": 85, "progressive_scans": 4}))
        m.append((f"{color}_opt", maker, size, color, {"quality": 85, "optimize_huffman": True}))
        m.append((f"{color}_rst", maker, size, color, {"quality": 85, "restart_interval": 7}))
    for hv in ((1, 1), (2, 1), (1, 2), (2, 2), (4, 1), (4, 2), (1, 4), (2, 4)):
        m.append((f"rgb_f{hv[0]}{hv[1]}", "ref_img_rgb", (258, 128), "rgb", {"quality": 90, "sampling": hv}))
        m.append((f"rgb_f{hv[0]}{hv[1]}_prog_opt_rst", "ref_img_rgb", (129, 67), "rgb",
                  {"quality": 75, "sampling": hv, "progressive_scans": 6, "optimize_huffman": True, "restart_interval": 5}))
    for kind in range(8):
        m.append((f"rgb_qt{kind}", "ref_img_rgb", (64, 48), "rgb", {"quality": 70, "qtables": (kind, kind)}))
    m.append(("bench_2000x1800", "bench_img", (2000, 1800), "rgb", {"quality": 90, "sampling": (2, 2)}))
    m.append(("one_pixel", "ref_img_rgb", (1, 1), "rgb", {"quality": 90}))
    m.append(("density_app", "ref_img_rgb", (33, 17), "rgb",
              {"quality": 90, "density": (1, 72, 96), "app_segments": [(2, bytes(range(40))), (15, b"x" * 300)]}))
    return m


def encode_case(case):
    import images
    from cases import oracle_encode
    name, maker, size, color, cfg = case
    return oracle_encode(getattr(images, maker)(*size), size[0], size[1], color, cfg)


def ints(text):
    return [int(x) for x in re.findall(r"-?\d+", text)]


def kat_rgb():
    src = open(os.path.join(REF, "image_buffer.rs")).read()
    out = []
    for mo in re.finditer(r"assert_rgb_to_ycbcr\(\[([^\]]*)\],\s*\[([^\]]*)\]\)", src):
        out.append(ints(mo.group(1)) + ints(mo.group(2)))
    return out


def kat_fdct():
    src = open(os.path.join(REF, "fdct.rs")).read()
    out = {}
    for mo in re.finditer(r"const (INPUT\d|OUTPUT\d): \[i16; 64\] = \[([^\]]*)\];", src):
        v = ints(mo.group(2))
        assert len(v) == 64
        out[mo.group(1)] = v
    return out


def reference_constants():
    def families(src, name):
        body = re.search(r"static " + name + r"[^=]*=\s*\[(.*?)\n\];", src, re.S).group(1)
        out = []
        for a in re.findall(r"\[([^\[\]]*?)\]", body, re.S):
            nums = ints(re.sub(r"//.*", "", a))
            if len(nums) == 64:
                out.append(nums)
        assert len(out) == 9, name
        return out

    def hex_array(src, name):
        return [int(x, 16) for x in re.findall(r"0x[0-9A-Fa-f]+", re.search(r"static " + name + r"[^=]*=\s*\[(.*?)\];", src, re.S).group(1))]

    quant = open(os.path.join(REF, "quantization.rs")).read()
    huff = open(os.path.join(REF, "huffman.rs")).read()
    writer = open(os.path.join(REF, "writer.rs")).read()
    return {
        "quantization_luma": families(quant, "DEFAULT_LUMA_TABLES"),
        "quantization_chroma": families(quant, "DEFAULT_CHROMA_TABLES"),
        "huffman": {k: {"counts": hex_array(huff, "DEFAULT_%s_CODE_LENGTHS" % k.upper()), "values": hex_array(huff, "DEFAULT_%s_VALUES" % k.upper())}
                    for k in ("luma_dc", "luma_ac", "chroma_dc", "chroma_ac")},
        "zigzag": ints(re.search(r"ZIGZAG[^=]*=\s*\[(.*?)\];", writer, re.S).group(1)),
    }


def write_reference_constants(consts):
    """one table per line"""
    s = json.dumps(consts, separators=(",", ":"))
    s = s.replace("],[", "],\n[").replace('{"', '{\n"').replace(',"', ',\n"')
    open(os.path.join(HERE, "reference_constants.json"), "w").write(s + "\n")


def main():
    if os.path.isdir(REF):
        write_reference_constants(reference_constants())
        rgb = kat_rgb()
        assert len(rgb) > 50
        json.dump(rgb, open(os.path.join(HERE, "rgb_to_ycbcr_kat.json"), "w"))
        f = kat_fdct()
        assert sorted(f) == ["INPUT1", "INPUT2", "OUTPUT1", "OUTPUT2"]
        json.dump(f, open(os.path.join(HERE, "fdct_kat.json"), "w"))
        print(f"KATs: {len(rgb)} colour triples, {len(f) // 2} DCT blocks")
    else:
        print("no /root/reference here: KAT files left as they are")
    hashes = {}
    for case in golden_matrix():
        data = encode_case(case)
        hashes[case[0]] = {"sha256": hashlib.sha256(data).hexdigest(), "len": len(data)}
    json.dump(hashes, open(os.path.join(HERE, "oracle_jpegs.json"), "w"), indent=0, sort_keys=True)
    print(f"oracle_jpegs.json: {len(hashes)} files")


if __name__ == "__main__":
    main()
