"""JPEG input (scope row f2): guetzli::Process(jpeg bytes), 4:4:4.  Fixtures are the
files under tests/golden/jpeg/ with the reference's answers in golden_jpeg.json
(tests/golden/make_golden_jpeg.py)."""
import hashlib
import json
import os

import pytest

import guetzli_b200 as gb
import parity
import refanswers

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = json.load(open(os.path.join(HERE, "golden", "golden_jpeg.json")))
# 4:2:0 input needs the YUV420 path (row f3): refused here, the reference accepts it
OUT_OF_SCOPE = {"sub420"}


def fixture(name):
    data = open(os.path.join(HERE, "golden", "jpeg", name + ".jpg"), "rb").read()
    assert hashlib.sha256(data).hexdigest() == GOLDEN[name]["input_sha256"]
    return data


def check_case(lib, name):
    g = GOLDEN[name]
    data = fixture(name)
    st = gb.ProcessStats(debug_output=[])
    p = gb.Params(butteraugli_target=gb.butteraugli_score_for_quality(g["quality"], lib=lib),
                  clear_metadata=g["clear_metadata"])
    ok, jpeg = gb.process_jpeg(p, st, data, lib=lib)
    if name in OUT_OF_SCOPE:
        assert not ok and jpeg == b""
        return
    assert ok == g["ok"], name
    assert len(jpeg) == g["jpeg_size"], f"{name}: {len(jpeg)} bytes vs {g['jpeg_size']}"
    assert hashlib.sha256(jpeg).hexdigest() == g["jpeg_sha256"], f"{name}: JPEG bytes differ"
    trace = "".join(st.debug_output)
    assert hashlib.sha256(trace.encode()).hexdigest() == g["trace_sha256"], f"{name}: verbose trace differs"
    assert [st.counters["number of iterations"], st.counters["number of iterations up"],
            st.counters["number of iterations down"]] == g["iterations"]


@pytest.mark.parametrize("name", sorted(GOLDEN))
def test_reader_matches_reference(port_lib, name):
    """ReadJpeg alone: accept / reject decision, geometry and every coefficient."""
    g = GOLDEN[name]
    ok, dims, coeffs = gb.api.read_jpeg(fixture(name), lib=port_lib)
    assert ok == g["read_ok"]
    if ok:
        assert dims == g["dims"]
        assert hashlib.sha256(coeffs.tobytes()).hexdigest() == g["coeffs_sha256"]


@pytest.mark.parametrize("name", ["base444_q90", "prog444_q85", "restart444_prog", "sub420", "gray", "odd444_prog",
                                  "meta_kept"])
def test_reader_differential_on_damaged_files(port_lib, ref, name):
    """Byte edits, bit flips and truncations of the fixtures: the parser must accept / reject and
    decode exactly like ReadJpeg."""
    import numpy as np
    rng = np.random.default_rng(sum(name.encode()))
    data = fixture(name)
    accepted = 0
    for t in range(60):
        b = bytearray(data)
        if t % 3 == 0:
            for _ in range(rng.integers(1, 4)):
                b[rng.integers(2, len(b))] = rng.integers(0, 256)
        elif t % 3 == 1:
            b[rng.integers(2, len(b))] ^= 1 << int(rng.integers(0, 8))
        else:
            b = b[:rng.integers(10, len(b))] + bytearray([0xff, 0xd9])
        rok, rdims, rcoeffs = ref.read_jpeg(bytes(b))
        ok, dims, coeffs = gb.api.read_jpeg(bytes(b), lib=port_lib)
        assert ok == rok, (name, t)
        if ok:
            accepted += 1
            assert dims == rdims and parity.same(coeffs, rcoeffs), (name, t)
    assert accepted > 0


@pytest.mark.parametrize("name", sorted(GOLDEN))
def test_port_process_jpeg_matches_golden(port_lib, name):
    check_case(port_lib, name)


def test_reference_reproduces_jpeg_golden(ref):
    for name in ("prog444_q85", "meta_kept", "tiny444", "gray"):
        g = GOLDEN[name]
        ok, jpeg, trace, counters = ref.process_jpeg(fixture(name), g["quality"], clear_metadata=g["clear_metadata"])
        assert ok == g["ok"] and refanswers.sha256(jpeg) == g["jpeg_sha256"]
        assert refanswers.sha256(trace) == g["trace_sha256"] and counters == g["iterations"]


def test_rgb_input_without_metadata_stripping(port_lib, ref):
    """Params::clear_metadata = false for RGB input: the encoder's own JFIF APP0 is the
    only metadata, so the output equals the stripped one (checked against the reference)."""
    from guetzli_b200 import synth
    rgb = synth.gradnoise(40, 48, 3)
    p = gb.Params(butteraugli_target=gb.butteraugli_score_for_quality(90, lib=port_lib), clear_metadata=False)
    ok, jpeg = gb.process(p, None, rgb, 48, 40, lib=port_lib)
    rok, rjpeg, _, _, _ = ref.process_rgb(rgb, 90, clear_metadata=False)
    assert ok and rok and rjpeg == jpeg and jpeg[2:4] == b"\xff\xe0"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["base444_q90", "prog444_q85", "noise444_q92", "odd444_prog", "restart444",
                                  "meta_kept", "tiny444_meta", "q100_tables1", "gray", "sub420", "truncated"])
def test_cuda_process_jpeg_matches_golden(cuda_lib, name):
    check_case(cuda_lib, name)
