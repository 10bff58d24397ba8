"""The tile layout with the first subsystem whole in the lane (TileLane<2,1,1>: 8 elements per lane, 4 trajectories per warp) on the
cnot2 example: against the CPU oracle, against the 2 x 2 tiles (TileLane<2,2>), and bit for bit across batch sizes and calls."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-10        # the reference's rule (test/evalGrad.jl), as in test_gpu_parity.py
TOL_22 = 1e-12     # the same sums in another order


def _rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300))


def _handle(cfg, inlane):
    import juqbox_b200 as jq
    old = os.environ.get("JQ_TILE_INLANE")
    os.environ["JQ_TILE_INLANE"] = inlane           # read when the handle is created
    try:
        wa = jq.Working_Arrays(cfg.params, cfg.nCoeff)
    finally:
        if old is None:
            os.environ.pop("JQ_TILE_INLANE")
        else:
            os.environ["JQ_TILE_INLANE"] = old
    wa.set_kernel(4)
    return wa


@pytest.fixture(scope="module")
def cnot2():
    from juqbox_b200 import configs
    return configs.example("cnot2")


@pytest.fixture(scope="module")
def inlane(cnot2):
    wa = _handle(cnot2, "1")
    yield wa
    wa.close()


@pytest.fixture(scope="module")
def tiles22(cnot2):
    wa = _handle(cnot2, "0")
    yield wa
    wa.close()


def _eval(wa, pc, tpc):
    r = wa.evaluate(pc)
    assert wa.last_kernel == 4 and wa.query(3) == tpc       # 16 trajectories per CTA: the in-lane tiles; 8: the 2 x 2 tiles
    return r


def test_inlane_matches_oracle(cnot2, inlane):
    from juqbox_b200 import configs
    from oracle import oracle_traceobjgrad
    nb = 5
    pc = configs.synthetic_pcof(cnot2, nb, seed_offset=3)
    pc[-1] = np.random.default_rng(17).uniform(-1, 1, cnot2.nCoeff) * cnot2.maxpar[0]      # full-amplitude stress vector
    o = oracle_traceobjgrad(cnot2.params, pc, None, nthreads=8)
    r = _eval(inlane, pc, 16)
    for k in ("infid", "leak"):
        assert np.all(np.abs(r[k] - o[k]) <= TOL * np.maximum(np.abs(o[k]), 1e-6)), (k, r[k], o[k])
    for b in range(nb):
        assert _rel(r["grad"][b, 0], o["grad"][b, 0]) < TOL, (b, _rel(r["grad"][b, 0], o["grad"][b, 0]))


def test_inlane_matches_2x2_tiles(cnot2, inlane, tiles22):
    from juqbox_b200 import configs
    pc = configs.synthetic_pcof(cnot2, 64, seed_offset=5) * 1.5
    a, b = _eval(inlane, pc, 16), _eval(tiles22, pc, 8)
    for k in ("infid", "leak", "trace_infid"):
        assert np.all(np.abs(a[k] - b[k]) <= TOL_22 * np.abs(b[k])), (k, np.max(np.abs(a[k] - b[k]) / np.abs(b[k])))
    for i in range(pc.shape[0]):
        assert _rel(a["grad"][i, 0], b["grad"][i, 0]) < TOL_22, (i, _rel(a["grad"][i, 0], b["grad"][i, 0]))


def test_inlane_ragged_batches_and_determinism(cnot2, inlane):
    """Four trajectories share a warp: a trajectory's results do not depend on its neighbours or on the batch size."""
    from juqbox_b200 import configs
    pc = configs.synthetic_pcof(cnot2, 4736 + 5, seed_offset=11)
    full = _eval(inlane, pc, 16)
    again = _eval(inlane, pc, 16)
    for k in ("infid", "leak", "trace_infid", "grad"):
        assert np.array_equal(full[k], again[k]), k
    for nb in (1, 3, 17):
        part = _eval(inlane, pc[-nb:], 16)
        for k in ("infid", "leak", "trace_infid", "grad"):
            assert np.array_equal(part[k], full[k][-nb:]), (k, nb)


def test_automatic_mode_switches_at_one_inlane_wave(cnot2):
    """Automatic mode takes the in-lane tiles from one full resident wave of them (2 CTAs of 16 trajectories per SM) and the
    2 x 2 tiles below it."""
    import torch
    import juqbox_b200 as jq
    from juqbox_b200 import configs
    wave = 2 * 16 * torch.cuda.get_device_properties(0).multi_processor_count
    pc = configs.synthetic_pcof(cnot2, wave, seed_offset=13)
    old = os.environ.pop("JQ_TILE_INLANE", None)
    try:
        wa = jq.Working_Arrays(cnot2.params, cnot2.nCoeff)
    finally:
        if old is not None:
            os.environ["JQ_TILE_INLANE"] = old
    try:
        full = _eval(wa, pc, 16)
        part = _eval(wa, pc[:wave - 1], 8)
        for k in ("infid", "grad"):
            assert np.max(np.abs(part[k] - full[k][:wave - 1])) <= TOL_22 * np.max(np.abs(full[k])), k
    finally:
        wa.close()
