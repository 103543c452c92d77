"""A slice of tools/fuzz_equivalence.py in the default suite: randomised models / optimizers / bucketing / accumulation /
re-bucketing / state-dict round trips on 2-4 ranks against single-process torch.optim."""
import importlib
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("seed", [3, 4])
def test_random_configurations_match_torch_optim(seed, monkeypatch):
    # the ranks unpickle the fuzzer's worker by module name: the module must be importable under its own name from a
    # path they inherit
    monkeypatch.syspath_prepend(os.path.join(ROOT, "tools"))
    fuzz = importlib.import_module("fuzz_equivalence")
    failures = fuzz.main(["--seed", str(seed), "--trials", "5", "--quiet"])
    assert not failures, failures[0]
