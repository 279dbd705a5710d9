"""GPU suite (-m gpu): the CUDA product, through its C ABI, against the oracle
(the unmodified reference, as its recorded answers: tests/refanswers.py)
and the committed golden answers.  Bit-exact everywhere: integers, float bit
patterns of every butteraugli stage, JPEG bytes and the verbose trace."""
import numpy as np
import pytest

import parity
from guetzli_b200 import synth

pytestmark = pytest.mark.gpu

SIZES = [(64, 96, 7), (70, 51, 3), (136, 200, 4)]


@pytest.mark.parametrize("h,w,seed", SIZES)
def test_integer_stages(cuda_lib, ref, h, w, seed):
    parity.check_integer_stages(cuda_lib, ref, synth.gradnoise(h, w, seed))


@pytest.mark.parametrize("h,w,seed", SIZES)
def test_butteraugli_stages(cuda_lib, ref, h, w, seed):
    parity.check_butteraugli_stages(cuda_lib, ref, synth.gradnoise(h, w, seed))


@pytest.mark.parametrize("h,w,seed", SIZES + [(40, 33, 2)])
def test_compare_and_block_kernels(cuda_lib, ref, h, w, seed):
    parity.check_compare_and_blocks(cuda_lib, ref, synth.noise(h, w, seed))


@pytest.mark.parametrize("h,w,seed", [(64, 96, 7), (40, 33, 2), (264, 520, 5)])
def test_device_save_jpeg(cuda_lib, ref, h, w, seed):
    parity.check_device_save_jpeg(cuda_lib, ref, synth.gradnoise(h, w, seed), seed)


@pytest.mark.parametrize("name", sorted(parity.GOLDEN))
def test_process_matches_golden(cuda_lib, name):
    st = parity.check_golden(cuda_lib, name)
    if not name.startswith("tiny"):
        assert st.device["gpu_launches"] > 0


def test_process_matches_reference_256(cuda_lib, ref):
    st = parity.check_process_vs_ref(cuda_lib, ref, synth.gradnoise(256, 256, 21), 92)
    assert st.device["gpu_launches"] > 0


@pytest.mark.parametrize("lookahead,new_model", [(3, False), (1, True), (5, False)])
def test_process_other_zeroing_params(cuda_lib, ref, lookahead, new_model):
    """zeroing_greedy_lookahead and the legacy zeroing score (processor.cc:391)."""
    parity.check_process_vs_ref(cuda_lib, ref, synth.gradnoise(96, 120, 12), 90, lookahead=lookahead,
                                new_zeroing_model=new_model)


def test_product_equals_port_on_512(cuda_lib, port_lib):
    """A larger case where the reference takes too long for a test: the CUDA
    product against the CPU restatement (itself pinned to the reference)."""
    rgb = synth.gradnoise(384, 512, 33)
    ok, jpeg, trace, _ = parity.run_process(cuda_lib, rgb, 90)
    ok2, jpeg2, trace2, _ = parity.run_process(port_lib, rgb, 90)
    assert ok and ok2 and trace == trace2 and jpeg == jpeg2


def test_full_size_properties_1080p(cuda_lib):
    """BASELINE config sizes, size-independent properties: (1) Compare of the
    unquantised image is deterministic across two contexts, (2) the distance is
    monotone under coarser quantisation, (3) scatter(restore) returns the exact
    distmap, (4) quantise is idempotent."""
    import guetzli_b200 as gb
    rgb = synth.gradnoise(1080, 1920, 4321)
    a = gb.DeviceImage(rgb, lib=cuda_lib)
    d0 = a.compare()
    dm0 = a.distmap()
    b = gb.DeviceImage(rgb, lib=cuda_lib)
    assert b.compare() == d0 and parity.bits_equal(b.distmap(), dm0)
    b.close()
    q2 = np.full((3, 64), 2, dtype=np.int32)
    q8 = np.full((3, 64), 8, dtype=np.int32)
    a.apply_global_quant(q2)
    c2 = a.download_candidate()
    d2 = a.compare()
    a.apply_global_quant(q8)
    d8 = a.compare()
    assert d0 <= d2 <= d8
    a.apply_global_quant(q2)
    assert np.array_equal(a.download_candidate(), c2)
    # zero a few coefficients then restore them: distmap must come back bit for bit
    dm2 = (a.compare(), a.distmap())
    flat = c2.reshape(-1)
    nz = np.flatnonzero(flat)[::5000][:200].astype(np.int32)
    a.scatter(nz, np.zeros(len(nz), dtype=np.int16))
    assert a.compare() >= 0
    a.scatter(nz, flat[nz])
    assert a.compare() == dm2[0] and parity.bits_equal(a.distmap(), dm2[1])
    a.close()


def _large_cases():
    import json
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_large.json")
    return json.load(open(path)) if os.path.exists(path) else {}


FULL_SIZE = {
    "noise1080p_s1234_q95": lambda: synth.noise(1080, 1920, 1234),          # BASELINE configs[1]
    "gradnoise4k_s4321_q90": lambda: synth.gradnoise(2160, 3840, 4321),     # configs[2]
    "gradnoise1024_s1000_q84": lambda: synth.gradnoise(1024, 1024, 1000),   # configs[4], image 0
    "gradnoise8k_s8192_q95": lambda: synth.gradnoise(4320, 7680, 8192),     # configs[3] (here: untiled, one GPU)
}


@pytest.mark.parametrize("name", [n for n in sorted(FULL_SIZE) if n in _large_cases()])
def test_process_matches_golden_full_size(cuda_lib, name):
    """BASELINE.json full-size configurations against the reference's own answers
    (tests/golden/make_golden_large.py: minutes to hours of CPU each)."""
    import hashlib
    g = _large_cases()[name]
    rgb = FULL_SIZE[name]()
    assert synth.sha256(rgb) == g["input_sha256"]
    ok, jpeg, trace, st = parity.run_process(cuda_lib, rgb, g["quality"])
    assert ok and len(jpeg) == g["jpeg_size"]
    assert hashlib.sha256(jpeg).hexdigest() == g["jpeg_sha256"]
    assert hashlib.sha256(trace.encode()).hexdigest() == g["trace_sha256"]
    assert [st.counters["number of iterations"], st.counters["number of iterations up"],
            st.counters["number of iterations down"]] == g["iterations"]


def test_batch64_matches_golden(cuda_lib):
    """BASELINE configs[4]: all 64 images gradnoise(1024, 1024, 1000 + i) at q84 against the
    reference's hashes (tests/golden/make_golden_batch64.sh), 16 at a time on this GPU."""
    import hashlib
    from concurrent.futures import ThreadPoolExecutor
    cases = _large_cases()
    names = ["gradnoise1024_s%d_q84" % (1000 + i) for i in range(64)]
    have = [n for n in names if n in cases]
    if len(have) < 64:
        pytest.skip("golden_large.json holds %d of the 64 batch answers" % len(have))

    def one(i):
        g = cases[names[i]]
        rgb = synth.gradnoise(1024, 1024, 1000 + i)
        assert synth.sha256(rgb) == g["input_sha256"]
        ok, jpeg, _, st = parity.run_process(cuda_lib, rgb, 84)
        return (ok, len(jpeg), hashlib.sha256(jpeg).hexdigest(), st.counters["number of iterations"])

    with ThreadPoolExecutor(16) as pool:
        got = list(pool.map(one, range(64)))
    for i, (ok, size, sha, iters) in enumerate(got):
        g = cases[names[i]]
        assert ok and size == g["jpeg_size"] and sha == g["jpeg_sha256"] and iters == g["iterations"][0], names[i]


def test_tiled_nccl_two_ranks():
    """BASELINE configs[3] plumbing on real hardware: ONE image over two ranks (one process per
    GPU, torchrun, the library's NCCL communicator), bytes equal to the reference's golden answer.
    Needs two GPUs; tests/run_tiled_nccl.py is the per-rank program."""
    import json
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    here = os.path.dirname(os.path.abspath(__file__))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29537", os.path.join(here, "run_tiled_nccl.py"), "bees"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    out = json.loads(line)
    assert out["world"] == 2 and out["bit_exact_vs_reference"]


AB_IMAGES = [("noise", 40, 33, 2), ("gradnoise", 70, 51, 3), ("noise", 136, 200, 4), ("gradnoise", 32, 300, 5),
             ("noise", 300, 32, 6), ("gradnoise", 260, 410, 8)]


@pytest.mark.parametrize("gen,h,w,seed", AB_IMAGES)
def test_fused_matches_staged(cuda_lib, gen, h, w, seed):
    """The TMA-staged fused Compare chain (fused_kernels.cuh, default) against the staged
    round-1 sequence of the same library (GB200_COMPARE=staged): every intermediate that both
    expose must have identical bits.  Localises a defect to a stage."""
    import os
    import guetzli_b200 as gb
    rgb = getattr(synth, gen)(h, w, seed)
    rng = np.random.default_rng(seed)
    plane = (rng.random((h, w), dtype=np.float32) * 255).astype(np.float32)
    q = parity.test_quant(seed)
    out = {}
    for mode in ("staged", "fused"):
        os.environ["GB200_COMPARE"] = mode
        try:
            img = gb.DeviceImage(rgb, lib=cuda_lib)
        finally:
            del os.environ["GB200_COMPARE"]
        r = {}
        for i in range(len(parity.BLUR_SPECS)):
            r["blur%d" % i] = img.debug_blur(plane, i)
        lin = img.debug_render()
        r["opsin"] = img.debug_opsin(lin)
        r["separate"] = img.debug_separate(r["opsin"])
        r["psycho0"] = img.debug_psycho0()
        r["corner_mask"] = img.debug_corner_mask()
        img.apply_global_quant(q)
        r["distance"] = np.float32(img.compare())
        r["distmap"] = img.distmap()
        r["weights"] = img.block_weights(-1, 2, 1.0, False)
        cand = img.download_candidate().reshape(-1)
        nz = np.flatnonzero(cand)[::7][:50].astype(np.int32)
        img.scatter(nz, np.zeros(len(nz), dtype=np.int16))
        r["distance2"] = np.float32(img.compare())
        r["distmap2"] = img.distmap()
        img.close()
        out[mode] = r
    for key in out["staged"]:
        a, b = np.asarray(out["staged"][key]), np.asarray(out["fused"][key])
        if not parity.bits_equal(a, b):
            bad = np.argwhere(a.view(np.uint32) != b.view(np.uint32))
            raise AssertionError(f"{key}: {len(bad)} of {a.size} values differ, first at {bad[0].tolist()}: "
                                 f"staged {a[tuple(bad[0])]!r} fused {b[tuple(bad[0])]!r}; "
                                 f"last at {bad[-1].tolist()}")


@pytest.mark.parametrize("name,world", [("bees_444x258_q95", 3), ("odd_70x51_s3_q88", 2)])
def test_strip_mode_on_one_gpu_matches_golden(cuda_lib, name, world):
    """Row-strip mode with the CUDA strip kernels (row-range launches, per-block
    exchange) driven by host threads that share this GPU: same bytes as untiled."""
    import hashlib
    import guetzli_b200 as gb
    g = parity.GOLDEN[name]
    rgb = parity.golden_input(name)
    h, w, _ = rgb.shape
    p = gb.Params(butteraugli_target=gb.butteraugli_score_for_quality(g["quality"], lib=cuda_lib))
    ok, jpeg = gb.process_tiled_threads(p, rgb, w, h, world, lib=cuda_lib)
    assert ok and hashlib.sha256(jpeg).hexdigest() == g["jpeg_sha256"]
