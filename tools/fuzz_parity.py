#!/usr/bin/env python3
"""Differential run of guetzli::Process(RGB) -- CPU port of the product's code against the unmodified
reference -- on random small images, qualities and zeroing parameters: JPEG bytes and --verbose trace must
be identical.  Test infrastructure (needs oracle/_ref and oracle/_build).
usage: tools/fuzz_parity.py [first_seed] [count]
environment: FUZZ_MAX_DIM (largest side, default 96), FUZZ_TILED=1 (also the strip mode over 2-6 thread ranks),
GB200_WALK=device / GB200_DEVICE_ORDER=1 (force the device half of the walk / the device replay of std::sort)"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import guetzli_b200 as gb  # noqa: E402
import reflib  # noqa: E402


def random_image(rng):
    top = int(os.environ.get("FUZZ_MAX_DIM", "96")) + 1  # larger images reach the device half of the walk more often
    h, w = int(rng.integers(32, top)), int(rng.integers(32, top))
    kind = int(rng.integers(0, 7))
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == 0:
        img = rng.integers(0, 256, (h, w, 3))
    elif kind == 1:   # smooth gradient + weak noise: long runs of equal walk keys
        img = np.stack([xx * 255 / (w - 1), yy * 255 / (h - 1), (xx + yy) * 255 / (w + h - 2)], -1) + rng.normal(0, 2, (h, w, 3))
    elif kind == 2:   # flat colour patches
        img = np.zeros((h, w, 3)) + rng.integers(0, 256, 3)
        img[h // 3:, w // 2:] = rng.integers(0, 256, 3)
    elif kind == 3:   # grayscale texture
        g = rng.integers(0, 256, (h, w))
        img = np.stack([g, g, g], -1)
    elif kind == 4:   # stripes / checkerboard with period 8: identical blocks (ties between blocks)
        img = np.where(((xx // 4 + yy // 4) % 2)[..., None] == 0, rng.integers(0, 256, 3), rng.integers(0, 256, 3))
    elif kind == 5:   # tiled copy of one random 16x16 patch
        p = rng.integers(0, 256, (16, 16, 3))
        img = np.tile(p, (h // 16 + 1, w // 16 + 1, 1))[:h, :w]
    else:             # saturated extremes
        img = rng.choice([0, 255], (h, w, 3)) * (rng.random((h, w, 1)) < 0.5) + rng.integers(0, 256, (h, w, 3)) * 0.1
    return np.clip(np.round(img), 0, 255).astype(np.uint8), kind


def one(seed, port, ref=reflib):
    rng = np.random.default_rng(seed)
    rgb, kind = random_image(rng)
    quality = float(rng.choice([84, 85, 88, 90, 93, 95, 97, 99, 100]))
    lookahead = int(rng.choice([1, 2, 3, 3, 3, 5]))
    new_model = bool(rng.random() < 0.8)
    rok, rjpeg, rtrace, _, _ = ref.process_rgb(rgb, quality, lookahead=lookahead, new_zeroing_model=new_model)
    h, w, _ = rgb.shape
    st = gb.ProcessStats(debug_output=[])
    p = gb.Params(butteraugli_target=gb.butteraugli_score_for_quality(quality, lib=port),
                  zeroing_greedy_lookahead=lookahead, new_zeroing_model=new_model)
    ok, jpeg = gb.process(p, st, rgb, w, h, lib=port)
    same = ok == rok and jpeg == rjpeg and "".join(st.debug_output) == rtrace
    if os.environ.get("FUZZ_TILED"):  # the row-strip mode (thread ranks) must give the same bytes
        world = int(rng.integers(2, 7))
        tok, tjpeg = gb.process_tiled_threads(p, rgb, w, h, world, lib=port)
        same = same and tok == ok and tjpeg == jpeg
    return same, dict(seed=seed, kind=kind, h=h, w=w, quality=quality, lookahead=lookahead, new_model=new_model,
                      iterations=st.counters.get("number of iterations"))


def main():
    first = int(sys.argv[1]) if len(sys.argv) > 1 else 0
    count = int(sys.argv[2]) if len(sys.argv) > 2 else 50
    port = gb.load_library(os.path.join(ROOT, "oracle", "_build", "libguetzli_port.so"))
    bad = 0
    for seed in range(first, first + count):
        same, info = one(seed, port)
        if not same:
            bad += 1
            print("MISMATCH", info, flush=True)
        if (seed - first + 1) % 25 == 0:
            print(f"... {seed - first + 1} cases, {bad} mismatches", flush=True)
    print(f"{count} cases from seed {first}: {bad} mismatches")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
