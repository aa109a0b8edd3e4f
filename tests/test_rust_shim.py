"""rust/ cannot be compiled in this image (no rustc/cargo), so the shim is checked as text: every public item of the
reference crate (src/lib.rs:45-49 and the signatures behind it, extracted by tests/golden/make_rust_api.py into
tests/golden/rust_public_api.json) must appear in rust/src/lib.rs with the same signature, every extern "C" declaration
must match include/jpegenc_b200.h, and the params struct must list the header's fields in the header's order."""
import json
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "rust_public_api.json")


def _norm(text):
    text = re.sub(r"//[^\n]*", "", text)
    text = re.sub(r"\s+", " ", text)
    return text.replace("( ", "(").replace(" )", ")").replace(",)", ")").replace("(mut self", "(self")


@pytest.fixture(scope="module")
def shim():
    return _norm(open(os.path.join(ROOT, "rust", "src", "lib.rs")).read())


@pytest.fixture(scope="module")
def api():
    return json.load(open(GOLD))


def _enum_body(shim, name):
    m = re.search(r"pub enum %s \{" % re.escape(name), shim)
    assert m, "enum %s missing" % name
    depth, i = 0, m.end() - 1
    j = i
    while True:
        if shim[j] == "{":
            depth += 1
        elif shim[j] == "}":
            depth -= 1
            if depth == 0:
                break
        j += 1
    return shim[i + 1:j]


def test_every_exported_item_exists(shim, api):
    for name in api["exports"]:
        assert re.search(r"pub (enum|struct|trait|fn) %s\b" % name, shim), "public item %s missing from the shim" % name


@pytest.mark.parametrize("enum", ["ColorType", "JpegColorType", "SamplingFactor", "QuantizationTableType", "PixelDensityUnit", "EncodingError"])
def test_enum_variants_in_reference_order(shim, api, enum):
    body = _enum_body(shim, enum)
    pos = -1
    for v in api[enum]:
        m = re.search(r"(?<![\w:])%s\b" % v, body[pos + 1:])
        assert m, "%s::%s missing or out of order" % (enum, v)
        pos += 1 + m.start()
    # no variant the reference does not have (user code that matches exhaustively must keep compiling)
    stripped = re.sub(r"\([^)]*\)|\{[^}]*\}|=[^,]*", "", re.sub(r"///[^\n]*", "", body))
    names = [t.strip() for t in stripped.split(",") if t.strip()]
    assert [re.match(r"\w+", n).group(0) for n in names] == api[enum]


def test_discriminants_are_the_abi_codes(shim):
    """ColorType is passed `as u8`: the shim's order must be include/jpegenc_b200.h's enum order."""
    hdr = open(os.path.join(ROOT, "include", "jpegenc_b200.h")).read()
    m = re.search(r"JPGB_LUMA = 0, JPGB_RGB = 1, JPGB_RGBA = 2, JPGB_BGR = 3, JPGB_BGRA = 4,\s*JPGB_YCBCR = 5, JPGB_CMYK = 6, JPGB_CMYK_AS_YCCK = 7, JPGB_YCCK = 8", hdr)
    assert m
    assert "Luma => 0, JpegColorType::Ycbcr => 5, JpegColorType::Cmyk => 6, JpegColorType::Ycck => 8" in shim


def test_method_signatures(shim, api):
    for key in ("Encoder", "Encoder<BufWriter<File>>", "SamplingFactor::fns", "PixelDensity::fns", "image_buffer::fns"):
        for sig in api[key]:
            assert _norm(sig) in shim, "signature missing or different: %s" % sig
    for key in ("ImageBuffer", "JfifWrite"):
        for sig in api[key]:
            assert _norm(sig) in shim, "trait method missing or different: %s" % sig
    for f in api["PixelDensity::fields"]:
        assert _norm(f) in shim


def test_error_impls_and_messages(shim, api):
    for imp in api["EncodingError::impls"]:
        assert re.search(r"impl %s for EncodingError" % re.escape(imp), shim), "impl %s for EncodingError missing" % imp
    for msg in api["EncodingError::display"]:
        assert '"%s"' % msg in shim, "Display text differs: %s" % msg
    assert "fn source(&self) -> Option<&(dyn Error + 'static)>" in shim


def test_extern_block_matches_the_c_header(shim):
    hdr = _norm(open(os.path.join(ROOT, "include", "jpegenc_b200.h")).read())
    ext = re.search(r'extern "C" \{(.*?)\} ', shim).group(1)
    fns = re.findall(r"fn (\w+)\(([^)]*)\)", ext)
    assert len(fns) >= 6
    for name, args in fns:
        m = re.search(r"\b%s\(([^)]*)\)" % name, hdr)
        assert m, "%s is not declared in include/jpegenc_b200.h" % name
        assert len([a for a in args.split(",") if a.strip()]) == len([a for a in m.group(1).split(",") if a.strip()]), name


def test_params_struct_field_order(shim):
    hdr = open(os.path.join(ROOT, "include", "jpegenc_b200.h")).read()
    body = re.search(r"typedef struct jpgb_params \{(.*?)\} jpgb_params;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    c_fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        for part in decl.split(","):
            c_fields.append(re.sub(r"\[.*", "", part.strip().split()[-1]).lstrip("*"))
    r_body = re.search(r"struct JpgbParams \{(.*?)\}", shim).group(1)
    r_fields = re.findall(r"(\w+):", r_body)
    assert r_fields == c_fields


def test_build_script_compiles_every_source():
    """rust/build.rs names each translation unit of csrc/ (a missing one is an unresolved symbol at cargo build time)"""
    import glob
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "rust", "build.rs")).read()
    src = glob.glob(os.path.join(root, "jpeg_encoder_b200", "csrc", "*.cu")) + glob.glob(os.path.join(root, "jpeg_encoder_b200", "csrc", "*.cpp"))
    assert src
    for s in src:
        assert '"%s"' % os.path.basename(s) in text, os.path.basename(s)
