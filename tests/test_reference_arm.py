# coding: utf-8
"""The oracle port against the unmodified reference package: same weights, same conditioning, same torch seed ->
torch.equal, so the "port" and "reference" kinds of bench.py's cpu_baseline compute the same thing.  What the
reference produced is stored under tests/golden/ by make_golden.py (reference_arm.npz: a short run with its own seed;
y_free of each case: the full-length run).  One copy runs in the CPU suite, one is marked gpu so that it also runs on
the host of the GPU machine.

The bench test times the reference package itself, which the repository cannot contain: __graft_entry__.build()
stages it under the git-ignored oracle/_ref/ where a checkout of it is available, and the test skips elsewhere."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, GOLDEN_DIR, ROOT
from helpers import GoldenCase
from oracle import wavenet_oracle as orc

REF_DIR = os.path.join(ROOT, "oracle", "_ref")
HAVE_REF = os.path.isfile(os.path.join(REF_DIR, "wavenet_vocoder", "wavenet.py"))
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="the reference package is not staged under oracle/_ref")


def check_case(name):
    gc = GoldenCase(name)
    cfg, w = gc.cfg, gc.w
    c_up, g_ids = gc.t("c_up"), gc.t("g_ids")
    g_vec = orc.embed_speaker(w, g_ids) if g_ids is not None else None
    short = np.load(os.path.join(GOLDEN_DIR, "reference_arm.npz"))
    y_ref = torch.from_numpy(short[name])
    T = y_ref.size(-1)
    with torch.no_grad():
        torch.manual_seed(int(short["seed"]))
        y_orc = orc.incremental_forward(cfg, w, c=None if c_up is None else c_up[..., :T], g=g_vec, T=T)
    assert torch.equal(y_ref, y_orc), name
    # and the full-length golden vector (seed of make_golden.py) is what the port produces from the torch seed alone
    with torch.no_grad():
        torch.manual_seed(gc.seed)
        y_full = orc.incremental_forward(cfg, w, c=c_up, g=g_vec, T=gc.T)
    ref = gc.t("y_free")
    if cfg.scalar_input:
        assert torch.equal(y_full, ref), name
    else:
        assert torch.equal(y_full.argmax(1), ref.long()), name


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_port_equals_staged_reference(name):
    check_case(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mol_cond", "gauss_speaker"])
def test_port_equals_staged_reference_on_gpu_box(name):
    check_case(name)


@needs_ref
def test_bench_reference_arm_uses_the_staged_package():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.load_reference() is not None
    m = bench.build_model()
    v, dt, n, kind = bench.time_cpu(m, 60, 5, 2, budget_s=2.0)
    assert kind == "reference" and v > 0 and n >= 50
