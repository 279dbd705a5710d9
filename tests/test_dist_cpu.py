"""World-size-2 gloo test of the sharded mode (one image per rank, no data-path
collective): the plumbing bench.py uses at N>1, driven on CPU with the port."""
import hashlib
import os
import socket
import sys

import numpy as np
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import time
    import guetzli_b200 as gb
    from guetzli_b200 import distributed as gdist, synth
    r, w, local, dist = gdist.setup("gloo")
    assert (r, w) == (rank, world)
    lib = gb.load_library(os.path.join(ROOT, "oracle", "_build", "libguetzli_port.so"))
    rgb = synth.gradnoise(48, 64, gdist.image_seed(100, r))
    params = gb.Params(butteraugli_target=gb.butteraugli_score_for_quality(90, lib=lib))
    gdist.barrier(dist, cuda=False)
    t0 = time.perf_counter()
    ok, jpeg = gb.process(params, None, rgb, 64, 48, lib=lib)
    dt = time.perf_counter() - t0
    assert ok
    gdist.barrier(dist, cuda=False)
    tmax = gdist.max_over_ranks(dist, dt)
    shas = gdist.gather_strings(dist, hashlib.sha256(jpeg).hexdigest(), w)
    assert tmax >= dt
    if r == 0:
        with open(os.path.join(out_dir, "result.txt"), "w") as f:
            f.write(" ".join(shas) + f" {gdist.throughput_mpix(w, 1, 48 * 64, tmax)}")
    dist.destroy_process_group()


def test_two_rank_sharded_run(tmp_path, port_lib, ref):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    parts = open(tmp_path / "result.txt").read().split()
    shas, mpix = parts[:world], float(parts[world])
    assert mpix > 0
    assert shas[0] != shas[1]  # distinct images per rank
    # every rank's output equals the reference's for that rank's image
    import refanswers
    from guetzli_b200 import synth
    for r in range(world):
        ok, jpeg, _, _, _ = ref.process_rgb(synth.gradnoise(48, 64, 100 + r), 90, trace=False)
        assert refanswers.sha256(jpeg) == shas[r]
