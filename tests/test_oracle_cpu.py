"""CPU suite (-m "not gpu"): pins the oracle.  The CPU restatement of the hot
path (oracle/_build/libguetzli_port.so, same kernel bodies as the CUDA product)
is checked against the unmodified reference (its recorded answers, tests/refanswers.py) stage by
stage and end to end, and against the committed golden answers."""
import os

import numpy as np
import pytest

import parity
from guetzli_b200 import synth

SIZES = [(64, 96, 7), (70, 51, 3)]


@pytest.mark.parametrize("h,w,seed", SIZES)
def test_port_integer_stages_match_reference(port_lib, ref, h, w, seed):
    parity.check_integer_stages(port_lib, ref, synth.gradnoise(h, w, seed))


@pytest.mark.parametrize("h,w,seed", SIZES)
def test_port_butteraugli_stages_match_reference(port_lib, ref, h, w, seed):
    parity.check_butteraugli_stages(port_lib, ref, synth.gradnoise(h, w, seed))


@pytest.mark.parametrize("h,w,seed", SIZES + [(40, 33, 2)])
def test_port_compare_and_block_kernels_match_reference(port_lib, ref, h, w, seed):
    parity.check_compare_and_blocks(port_lib, ref, synth.noise(h, w, seed))


@pytest.mark.parametrize("name", [n for n in parity.GOLDEN if not n.startswith("bees")])
def test_port_process_matches_golden(port_lib, name):
    parity.check_golden(port_lib, name)


def test_port_process_bees_matches_golden(port_lib):
    """BASELINE.json configs[0]: tests/bees.png --quality 95."""
    parity.check_golden(port_lib, "bees_444x258_q95")


def test_reference_reproduces_golden(ref):
    """The committed golden answers are what the reference produces."""
    import refanswers
    for name in ("gradnoise_64x96_s7_q90", "gray_64x64_s9_q90"):
        g = parity.GOLDEN[name]
        ok, jpeg, trace, cnt, _ = ref.process_rgb(parity.golden_input(name), g["quality"])
        assert refanswers.sha256(jpeg) == g["jpeg_sha256"]
        assert cnt == g["iterations"]


def test_tables_match_reference(port_lib, ref):
    """Generated / formula tables equal the reference's literal tables."""
    cr_r, cb_b, cr_g, cb_g, rl = ref.color_tables()
    x = np.arange(256) - 128
    assert parity.same((91881 * x + 32768) >> 16, cr_r)
    assert parity.same((116130 * x + 32768) >> 16, cb_b)
    assert parity.same(-46802 * x, cr_g)
    assert parity.same(-22554 * x + 32768, cb_g)
    assert parity.same(np.clip(np.arange(1024) - 384, 0, 255).astype(np.uint8), rl)
    for q in (84, 90, 95, 97.5, 100, 110, 60):
        assert port_lib.gb200_butteraugli_score_for_quality(float(q)) == ref.score_for_quality(float(q))


def test_rejects_low_quality_and_bad_sizes(port_lib):
    import guetzli_b200 as gb
    rgb = synth.gradnoise(40, 40, 1)
    p = gb.Params(butteraugli_target=gb.butteraugli_score_for_quality(80, lib=port_lib))
    ok, jpeg = gb.process(p, None, rgb, 40, 40, lib=port_lib)
    assert not ok and jpeg == b""            # quality < 84 (processor.cc:800)
    ok, jpeg = gb.process(gb.Params(), None, rgb, 41, 40, lib=port_lib)
    assert not ok and jpeg == b""            # rgb.size() != 3*w*h (jpeg_data_encoder.cc:68)
    ok, jpeg = gb.process(gb.Params(force_420=True), None, rgb, 40, 40, lib=port_lib)
    assert not ok                            # YUV420 is out of scope


@pytest.mark.parametrize("lookahead,new_model", [(3, False), (1, True), (5, True), (2, False)])
def test_port_process_other_zeroing_params(port_lib, ref, lookahead, new_model):
    """Params::zeroing_greedy_lookahead / new_zeroing_model (processor.h:35-36; the
    legacy score of processor.cc:391-392) against the reference itself."""
    rgb = synth.gradnoise(48, 56, 11)
    parity.check_process_vs_ref(port_lib, ref, rgb, 90, lookahead=lookahead, new_zeroing_model=new_model)


def test_partial_order_is_arrangement_independent(port_lib, ref, monkeypatch):
    """The device returns the smallest walk-order keys in arbitrary order and equal
    keys may be arranged differently from the reference's std::sort.  The result must
    not depend on that: noise images are rich in equal keys; shuffle the fetched
    entries (test hook of the CPU port) and compare with the reference."""
    rgb = synth.noise(160, 224, 77)
    rok, rjpeg, rtrace, _, _ = ref.process_rgb(rgb, 95)
    for seed in ("1", "2"):
        monkeypatch.setenv("GB200_SHUFFLE_ORDER", seed)
        ok, jpeg, trace, st = parity.run_process(port_lib, rgb, 95)
        assert st.device["order_partial"] > 50
        assert trace == rtrace and jpeg == rjpeg


def test_refusals_are_pinned(port_lib, capfd):
    """What this implementation refuses although the reference accepts it (YUV420, DESIGN.md
    "Out of scope") and what it refuses for its own limits, with the exact messages the CLI
    usage text and README quote."""
    import guetzli_b200 as gb
    rgb = synth.gradnoise(40, 40, 1)
    for kw in ({"try_420": True}, {"force_420": True}):
        p = gb.Params(butteraugli_target=1.0, **kw)
        ok, jpeg = gb.process(p, None, rgb, 40, 40, lib=port_lib)
        assert not ok and jpeg == b""
        assert "guetzli_b200: YUV420 is outside the B200 hot path (DESIGN.md)" in capfd.readouterr().err
    jpg420 = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "jpeg", "sub420.jpg"), "rb").read()
    ok, jpeg = gb.process_jpeg(gb.Params(butteraugli_target=1.0), None, jpg420, lib=port_lib)
    assert not ok and jpeg == b""
    assert "YUV420 JPEG input is outside the B200 hot path" in capfd.readouterr().err
    # 32-bit device indices: refused up front, nothing allocated
    big = np.zeros(3 * 65535 * 4, dtype=np.uint8)  # the size check comes before the buffer is read
    import ctypes as C
    from guetzli_b200.api import _CParams, _CStats, _LOG_FN
    cp = _CParams(1.0, 1, 0, 0, 0, 3, 1)
    out, out_len, cs = C.POINTER(C.c_uint8)(), C.c_size_t(), _CStats()
    ok = port_lib.gb200_process_rgb(C.byref(cp), big.ctypes.data, 65535, 65535, 0, C.cast(None, _LOG_FN), None,
                                    C.byref(out), C.byref(out_len), C.byref(cs))
    assert not ok and out_len.value == 0
    assert "image too large (65535 x 65535)" in capfd.readouterr().err


def test_port_device_walk(port_lib, ref, monkeypatch):
    """The device half of the selection walk (walk_dev.h: two-rank radix select, bulk applied
    as a set, host loop on the window only) through the CPU port's emulated kernels, with the
    device's symbol histograms checked against the host's every iteration."""
    monkeypatch.setenv("GB200_WALK", "device")
    monkeypatch.setenv("GB200_CHECK_HOST_HIST", "1")
    for rgb, q in ((synth.noise(160, 224, 77), 95), (synth.gradnoise(192, 256, 5), 90)):
        rok, rjpeg, rtrace, _, _ = ref.process_rgb(rgb, q)
        ok, jpeg, trace, st = parity.run_process(port_lib, rgb, q)
        assert ok == rok and trace == rtrace and jpeg == rjpeg


def test_process_is_reentrant(port_lib):
    """Process() from several host threads at once (one context + stream per call, the
    batch mode of bench.py): every result equals the sequential one."""
    from concurrent.futures import ThreadPoolExecutor
    jobs = [(synth.gradnoise(40 + 8 * i, 48, 20 + i), 88 + i) for i in range(6)]
    jobs.append((synth.noise(24, 40, 3), 95))   # below 32 px: no search
    seq = [parity.run_process(port_lib, rgb, q)[:3] for rgb, q in jobs]
    with ThreadPoolExecutor(4) as pool:
        par = list(pool.map(lambda j: parity.run_process(port_lib, j[0], j[1])[:3], jobs * 2))
    assert par == seq + seq


def test_repeated_blocks_tie_everywhere(port_lib, ref):
    """An image made of two copies of the same noise tile: every block has a twin with
    bit-identical candidate errors, so the global order is full of equal keys of
    different blocks.  The device top-K path must notice where the arrangement of such
    runs matters (and then take the reference-ordered sort) and still end up with the
    reference's bytes and trace."""
    import numpy as np
    rgb = np.ascontiguousarray(np.tile(synth.noise(112, 112, 11), (1, 2, 1)))
    st = parity.check_process_vs_ref(port_lib, ref, rgb, 94)
    assert st.device["order_exact"] > 100 and st.device["order_partial"] > 50


def test_huffman_code_lengths_match_reference(port_lib, ref):
    """The sort-once builder of the code lengths (jpeg_out.cc huffman_code_lengths) against the
    reference's CreateHuffmanTree (guetzli/entropy_encode.cc:73) on histograms that need anywhere
    from one to many count floors, incl. ties, single symbols and the phantom symbol 256."""
    import ctypes as C
    port_lib.gb200_debug_huffman_depths.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    port_lib.gb200_debug_huffman_depths.restype = None
    rng = np.random.default_rng(77)
    n = 257
    trials = 3000
    all_counts = np.zeros((trials, n), dtype=np.uint32)
    limits = np.zeros(trials, dtype=np.int32)
    mine = np.zeros((trials, n), dtype=np.uint8)
    for t in range(trials):
        mode = t % 7
        present = rng.random(n) < rng.uniform(0.02, 1.0)
        if mode == 0:
            c = rng.integers(1, 5, n)
        elif mode == 1:
            c = 1 << rng.integers(0, 28, n)
        elif mode == 2:
            c = rng.integers(1, 1 << int(rng.integers(2, 25)), n)
        elif mode == 3:
            c = 2 * rng.integers(1, 1000, n)
        elif mode == 4:
            c = np.where(rng.random(n) < 0.3, 1, rng.integers(1, 5_000_000, n))
        elif mode == 5:
            c = (1 + 4_000_000 * rng.random(n) ** 8).astype(np.int64)
        else:  # Fibonacci-like counts: the deepest possible trees
            c = np.ones(n, dtype=np.int64)
            f = [1, 1]
            while len(f) < 40:
                f.append(f[-1] + f[-2])
            idx = rng.permutation(n)[:40]
            c[idx] = np.array(f[:40], dtype=np.int64)
            present[idx] = True
        counts = np.where(present, c, 0).astype(np.uint32)
        counts[256] = 1
        limits[t] = 12 if t % 11 == 0 else 16
        all_counts[t] = counts
        port_lib.gb200_debug_huffman_depths(counts.ctypes.data, n, int(limits[t]), mine[t].ctypes.data)
    theirs = ref.huffman_depths(all_counts, limits)
    if not parity.same(mine, theirs):
        bad = [t for t in range(trials) if not np.array_equal(mine[t], theirs[t])] if isinstance(theirs, np.ndarray) else []
        raise AssertionError(f"code lengths differ from the reference's (trials {bad[:10]}, mode = trial % 7)")


@pytest.mark.parametrize("h,w,seed", [(64, 96, 7), (40, 33, 2), (72, 136, 5)])
def test_port_device_save_jpeg(port_lib, ref, h, w, seed):
    parity.check_device_save_jpeg(port_lib, ref, synth.gradnoise(h, w, seed), seed)


def test_420_flags_where_the_reference_does_not_downsample(port_lib, ref):
    """Params::try_420 on a grayscale image (IsGrayscale, processor.cc:782,846), try_420 / force_420 on an
    image too small for Butteraugli (:832-838) and force_420 on a grayscale image (nothing to downsample,
    output_image.cc:305) never subsample anything in the reference: same bytes and trace as the reference
    run with the same flags."""
    cases = [(parity.gray(64, 64, 9), 90, dict(try_420=True)),
             (synth.gradnoise(20, 40, 5), 95, dict(force_420=True)),
             (synth.gradnoise(20, 40, 5), 95, dict(try_420=True)),
             # force_420 on a grayscale image: the YUV420 pass with nothing to downsample (one-component
             # JPEGData, quant search from score 0, masking of component 0 with a single AC histogram)
             (parity.gray(64, 64, 9), 90, dict(force_420=True)),
             (parity.gray(48, 72, 3), 95, dict(force_420=True, try_420=True)),
             (np.full((40, 40, 3), 77, dtype=np.uint8), 95, dict(force_420=True))]
    for rgb, quality, flags in cases:
        rok, rjpeg, rtrace, _, _ = ref.process_rgb(rgb, quality, **flags)
        ok, jpeg, trace, _ = parity.run_process(port_lib, rgb, quality, **flags)
        assert ok and rok and jpeg == rjpeg and trace == rtrace, flags
