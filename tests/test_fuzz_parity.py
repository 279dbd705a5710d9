"""A fixed handful of cases of tools/fuzz_parity.py (random small images, qualities and zeroing
parameters; CPU port of the product's code vs the unmodified reference, bytes + trace)."""
import importlib.util
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("fuzz_parity", os.path.join(ROOT, "tools", "fuzz_parity.py"))
fuzz = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(fuzz)


@pytest.mark.parametrize("seed", [3, 11, 19, 24, 30, 37, 1012, 2044])
def test_random_case_matches_reference(port_lib, ref, seed):
    same, info = fuzz.one(seed, port_lib, ref)
    assert same, info


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [3, 19, 30, 1012])
def test_random_case_matches_reference_cuda(cuda_lib, ref, seed):
    same, info = fuzz.one(seed, cuda_lib, ref)
    assert same, info
