"""Stage-by-stage and end-to-end parity checks shared by the CPU-port tests
(oracle pinning) and the GPU tests (product vs oracle).  `lib` is a C-ABI
library handle (product or port); `ref` answers like tests/reflib (the real reference), live or
as its recorded answers (tests/refanswers.py)."""
import hashlib
import json
import os

import numpy as np

import guetzli_b200 as gb
from guetzli_b200 import synth
from refanswers import Digest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = json.load(open(os.path.join(HERE, "golden", "golden.json")))

BLUR_SPECS = [(1.2, 0.0), (7.46953768697, -0.00457628248637), (3.734768843485, -0.271277366628),
              (1.8673844217425, 0.147068973249), (10.6666499623, 0.0),
              (9.24456601467, -0.0724948220913), (2.3770330432, -0.0724948220913),
              (9.04353323561, -0.0724948220913), (1.72547472444, 1.0)]


def bits_equal(a, b):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if isinstance(b, Digest):
        return b == a
    b = np.ascontiguousarray(b, dtype=np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def same(a, b):
    """np.array_equal(a, b) where b is the reference's answer (an array or its Digest)."""
    return b == a if isinstance(b, Digest) else np.array_equal(a, b)


def gray(h, w, seed):
    g = synth.gradnoise(h, w, seed)[..., 1]
    return np.stack([g, g, g], axis=-1)


def golden_input(name):
    if name.startswith("bees"):
        return np.load(os.path.join(HERE, "golden", "bees_rgb.npz"))["rgb"]
    table = {
        "gradnoise_64x96_s7_q90": lambda: synth.gradnoise(64, 96, 7),
        "noise_48x40_s5_q95": lambda: synth.noise(48, 40, 5),
        "tiny_20x40_s5_q95": lambda: synth.gradnoise(20, 40, 5),
        "odd_70x51_s3_q88": lambda: synth.gradnoise(70, 51, 3),
        "gray_64x64_s9_q90": lambda: gray(64, 64, 9),
        "gradnoise_128x128_s11_q84": lambda: synth.gradnoise(128, 128, 11),
        "min_32x32_s2_q90": lambda: synth.noise(32, 32, 2),
        "small_33x47_s4_q95": lambda: synth.gradnoise(33, 47, 4),
        "wide_32x200_s6_q88": lambda: synth.gradnoise(32, 200, 6),
        "flat_40x40_q95": lambda: np.full((40, 40, 3), 77, dtype=np.uint8),
    }
    return table[name]()


def test_quant(seed=0):
    rng = np.random.default_rng(seed)
    q = rng.integers(1, 12, (3, 64)).astype(np.int32)
    q[:, 0] = rng.integers(1, 4, 3)
    return q


def check_integer_stages(lib, ref, rgb):
    """a2 FDCT, a8 quantise, a7+a9 render: bit-exact integers / float LUT values."""
    h, w, _ = rgb.shape
    img = gb.DeviceImage(rgb, lib=lib)
    ref_c = ref.rgb_to_coeffs(rgb)
    assert same(img.orig_coeffs(), ref_c), "FDCT coefficients differ"
    q = test_quant(1)
    cq = ref.apply_global_quant(ref_c, w, h, q)
    img.apply_global_quant(q)
    assert same(img.download_candidate(), cq), "global quantisation differs"
    _, lin = ref.render(cq, w, h)
    assert bits_equal(img.debug_render(), lin), "rendered linear RGB differs"
    img.close()


def check_butteraugli_stages(lib, ref, rgb):
    """blur x9, render, opsin, frequency split: bit-identical floats.  Each stage gets the
    library's output of the stage before, once that is checked against the reference's."""
    h, w, _ = rgb.shape
    img = gb.DeviceImage(rgb, lib=lib)
    rng = np.random.default_rng(1)
    plane = (rng.random((h, w), dtype=np.float32) * 255).astype(np.float32)
    for i, (s, b) in enumerate(BLUR_SPECS):
        assert bits_equal(img.debug_blur(plane, i), ref.blur(plane, s, b)), f"blur {i} differs"
    _, lin_ref = ref.render(ref.rgb_to_coeffs(rgb), w, h)
    lin = img.debug_render()
    assert bits_equal(lin, lin_ref), "rendered linear RGB differs"
    xyb = img.debug_opsin(lin)
    assert bits_equal(xyb, ref.opsin(lin)), "opsin differs"
    assert bits_equal(img.debug_separate(xyb), ref.separate(xyb)), "frequency split differs"
    img.close()


def check_compare_and_blocks(lib, ref, rgb, target=0.9):
    """a10 Compare (distmap + distance), a13 masks, a15 weights, a14 zeroing orders, a11 JPEG bytes."""
    h, w, _ = rgb.shape
    img = gb.DeviceImage(rgb, lib=lib)
    ref_c = ref.rgb_to_coeffs(rgb)
    q = test_quant(2)
    cq = ref.apply_global_quant(ref_c, w, h, q)
    img.apply_global_quant(q)
    cand = img.download_candidate()
    assert same(cand, cq), "global quantisation differs"
    dist = img.compare()
    rdm, rdist = ref.compare_coeffs(rgb, cq, target)
    assert dist == rdist, f"distance {dist} vs {rdist}"
    assert bits_equal(img.distmap(), rdm), "distmap differs"
    assert bits_equal(img.debug_corner_mask(), ref.block_corner_mask(rgb)), "block-corner mask differs"
    for d, r, z in [(1, 1, True), (1, 2, False), (-1, 1, False), (-1, 4, False)]:
        mine = img.block_weights(d, r, target * 1.0, z)
        theirs = ref.block_weights(w, h, target, d, r, 1.0, np.zeros((h, w), dtype=np.float32) if z else rdm)
        assert same(mine, theirs), f"block weights differ (dir {d}, r {r})"
    idx, err, cnt = img.zeroing_orders(target, 3)
    roffs, ridx, rerr = ref.zeroing_orders(rgb, ref_c, q, target)
    # the reference's lists of all blocks back to back, from offsets roffs
    assert same(np.concatenate([[0], np.cumsum(cnt)]), roffs), "zeroing-order list lengths differ"
    assert same(np.concatenate([idx[b, :n] for b, n in enumerate(cnt)]), ridx), "zeroing orders differ"
    assert bits_equal(np.concatenate([err[b, :n] for b, n in enumerate(cnt)]), rerr), "zeroing-order errors differ"
    assert gb.write_jpeg(cand, w, h, q, lib=lib) == ref.write_jpeg(ref_c, w, h, q), "JPEG bytes differ"
    img.close()


def run_process(lib, rgb, quality, device=0, **params):
    h, w, _ = rgb.shape
    st = gb.ProcessStats(debug_output=[])
    p = gb.Params(butteraugli_target=gb.butteraugli_score_for_quality(quality, lib=lib), **params)
    ok, jpeg = gb.process(p, st, rgb, w, h, device=device, lib=lib)
    return ok, jpeg, "".join(st.debug_output), st


def check_golden(lib, name):
    """guetzli::Process(RGB) against the committed known answers of the reference."""
    g = GOLDEN[name]
    rgb = golden_input(name)
    assert synth.sha256(rgb) == g["input_sha256"], "input generator drifted"
    ok, jpeg, trace, st = run_process(lib, rgb, g["quality"])
    assert ok == g["ok"]
    assert len(jpeg) == g["jpeg_size"], f"{name}: {len(jpeg)} bytes vs {g['jpeg_size']}"
    assert hashlib.sha256(jpeg).hexdigest() == g["jpeg_sha256"], f"{name}: JPEG bytes differ"
    assert hashlib.sha256(trace.encode()).hexdigest() == g["trace_sha256"], f"{name}: verbose trace differs"
    assert [st.counters["number of iterations"], st.counters["number of iterations up"],
            st.counters["number of iterations down"]] == g["iterations"]
    return st


def check_process_vs_ref(lib, ref, rgb, quality, lookahead=3, new_zeroing_model=True):
    ok, jpeg, trace, st = run_process(lib, rgb, quality, zeroing_greedy_lookahead=lookahead,
                                      new_zeroing_model=new_zeroing_model)
    rok, rjpeg, rtrace, rcnt, _ = ref.process_rgb(rgb, quality, lookahead=lookahead,
                                                  new_zeroing_model=new_zeroing_model)
    assert ok == rok
    if trace != rtrace and isinstance(rtrace, str):
        a, b = trace.split("\n"), rtrace.split("\n")
        for i, (x, y) in enumerate(zip(a, b)):
            assert x == y, f"trace line {i}:\n  mine: {x}\n  ref : {y}"
    assert trace == rtrace, "verbose trace differs"
    assert jpeg == rjpeg, "JPEG bytes differ"
    return st


def adversarial_candidates(nblocks, q, seed):
    """Candidate coefficient sets (multiples of q) that stress the entropy coder: zero runs of 16 and
    more (ZRL), a lone last coefficient, all-zero blocks, the largest magnitudes the device quotient
    supports, DC swings, zero chroma (one-component output), dense random blocks."""
    rng = np.random.default_rng(seed)
    zz = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                   7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38,
                   31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63])
    q = np.asarray(q, dtype=np.int64).reshape(3, 64)
    out = {}
    # sparse: few nonzero coefficients far apart in zig-zag order -> ZRL symbols, end-of-block after a run
    lv = np.zeros((3, nblocks, 64), dtype=np.int64)
    for c in range(3):
        for b in range(nblocks):
            for z in rng.choice(np.arange(1, 64), size=int(rng.integers(0, 4)), replace=False):
                lv[c, b, zz[z]] = int(rng.integers(-3, 4))
            lv[c, b, 0] = int(rng.integers(-40, 41))
    lv[0, : max(1, nblocks // 7), 1:] = 0          # DC-only blocks
    lv[:, nblocks // 2, :] = 0                      # an all-zero MCU
    lv[0, nblocks - 1, 1:] = 0
    lv[0, nblocks - 1, 63] = 1                      # a lone coefficient at the very end: three ZRLs, no EOB
    out["sparse"] = lv
    # dense random levels incl. large magnitudes (|level * q| stays below 2^15)
    lim = np.minimum(1023, 32767 // q)[:, None, :]
    dense = rng.integers(-1023, 1024, (3, nblocks, 64))
    dense = np.clip(dense, -lim, lim)
    dense[:, :, 1:] = np.where(rng.random((3, nblocks, 63)) < 0.35, 0, dense[:, :, 1:])
    out["dense"] = dense
    # luma only: both chroma components zero -> a one-component file
    gray = dense.copy()
    gray[1:] = 0
    out["gray"] = gray
    # extreme DC differences
    swing = np.zeros((3, nblocks, 64), dtype=np.int64)
    swing[:, ::2, 0] = lim[:, 0, 0][:, None]
    swing[:, 1::2, 0] = -lim[:, 0, 0][:, None]
    out["dc_swing"] = swing
    return {k: (v * q[:, None, :]).astype(np.int16) for k, v in out.items()}


def check_device_save_jpeg(lib, ref, rgb, seed=0):
    """a11 + f1 as one call (gb200_image_save_jpeg): the device's file equals the reference's
    SaveToJpegData + WriteJpeg (and the host serialiser) on coefficient patterns that natural images rarely have."""
    h, w, _ = rgb.shape
    q = test_quant(seed)
    img = gb.DeviceImage(rgb, lib=lib)
    try:
        img.apply_global_quant(q)
        cases = {"quantised_original": img.download_candidate()}
        cases.update(adversarial_candidates(img.nblocks, q, seed))
        for name, coeffs in cases.items():
            img.upload_candidate(coeffs)
            got = img.save_jpeg(q)
            want = ref.write_jpeg(coeffs, w, h, q)
            assert got == want, (name, len(got))
            assert got == gb.write_jpeg(coeffs, w, h, q, lib=lib), name
    finally:
        img.close()
