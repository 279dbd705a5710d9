"""Stand-alone butteraugli (scope row f4): gb200_butteraugli_diffmap and the `butteraugli`
command line against butteraugli::ButteraugliInterface / CreateHeatMapImage of the
reference (its recorded answers, tests/refanswers.py), bit for bit."""
import os
import subprocess

import numpy as np
import pytest
from PIL import Image

import guetzli_b200 as gb
import parity
from guetzli_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI_PORT = os.path.join(ROOT, "oracle", "_build", "butteraugli_port")
CLI = os.path.join(ROOT, "guetzli_b200", "butteraugli")

# butteraugli_main.cc:137: the tool's own sRGB -> linear table
_TABLE = np.array([255.0 * ((i / 255.0) / 12.92 if i / 255.0 <= 0.04045 else ((i / 255.0 + 0.055) / 1.055) ** 2.4)
                   for i in range(256)])


def linear(rgb):
    return np.ascontiguousarray(_TABLE[rgb].transpose(2, 0, 1)).astype(np.float32)


def pair(h, w, seed):
    a = synth.noise(h, w, seed) // 2 + 64
    b = np.clip(a.astype(int) + synth.noise(h, w, seed + 1) % 9 - 4, 0, 255).astype(np.uint8)
    return a.astype(np.uint8), b


SIZES = [(40, 56), (8, 8), (5, 20), (3, 3), (33, 9), (1, 1), (17, 130), (64, 64)]


def check_api(lib, ref, h, w):
    a, b = pair(h, w, 10 * h + w)
    d0, s0 = ref.butteraugli_interface(linear(a), linear(b))
    d1, s1 = gb.api.butteraugli_diffmap(linear(a), linear(b), lib=lib)
    assert s0 == s1 and parity.bits_equal(d1, d0), (h, w)
    # identical images: zero everywhere
    d2, s2 = gb.api.butteraugli_diffmap(linear(a), linear(a), lib=lib)
    assert s2 == 0.0 and not d2.any()


def check_cli(cli, ref, tmp_path):
    a, b = pair(48, 40, 77)
    pa, pb, hm = str(tmp_path / "a.png"), str(tmp_path / "b.png"), str(tmp_path / "heat.ppm")
    Image.fromarray(a).save(pa)
    Image.fromarray(b).save(pb)
    r = subprocess.run([cli, pa, pb, hm], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr
    d0, s0 = ref.butteraugli_interface(linear(a), linear(b))
    assert r.stdout.decode() == "%f\n" % s0
    header = b"P6\n40 48\n255\n"
    ppm = open(hm, "rb").read()
    assert ppm[:len(header)] == header and len(ppm) == len(header) + 48 * 40 * 3
    assert parity.same(np.frombuffer(ppm[len(header):], dtype=np.uint8).reshape(48, 40, 3), ref.heatmap(d0))
    # RGBA: scored over black and over white, the larger distance is reported
    alpha = (synth.noise(48, 40, 5)[..., 0] // 64 * 85).astype(np.uint8)
    Image.fromarray(np.dstack([a, alpha])).save(pa)
    Image.fromarray(np.dstack([b, alpha])).save(pb)
    r = subprocess.run([cli, pa, pb], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr

    def over(rgb, bg):
        al = alpha.astype(int)[..., None]
        v = (rgb.astype(int) * al + bg * (255 - al) + 127) // 255
        v = np.where(al == 255, rgb, np.where(al == 0, bg, v))
        return linear(v.astype(np.uint8))
    want = max(ref.butteraugli_interface(over(a, bg), over(b, bg))[1] for bg in (0, 255))
    assert r.stdout.decode() == "%f\n" % want
    # failures
    assert subprocess.run([cli, pa], stderr=subprocess.PIPE).returncode == 1
    Image.fromarray(a[:20]).save(pb)
    assert subprocess.run([cli, pa, pb], stderr=subprocess.PIPE).returncode == 1
    assert subprocess.run([cli, pa, os.devnull], stderr=subprocess.PIPE).returncode == 1


@pytest.mark.parametrize("h,w", SIZES)
def test_port_diffmap_matches_reference(port_lib, ref, h, w):
    check_api(port_lib, ref, h, w)


def test_port_cli(port_lib, ref, tmp_path):
    check_cli(CLI_PORT, ref, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", SIZES + [(300, 411)])
def test_cuda_diffmap_matches_reference(cuda_lib, ref, h, w):
    check_api(cuda_lib, ref, h, w)


@pytest.mark.gpu
def test_cuda_cli(cuda_lib, ref, tmp_path):
    check_cli(CLI, ref, tmp_path)
