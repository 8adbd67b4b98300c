"""GPU == GPU: our engine against the UNMODIFIED reference GPU path on the same cuRAND seed.

The reference side is stored under tests/golden/reference_gpu/ (tests/golden/make_reference_gpu.py): what the reference's
own VanillaMPPIController + kernels (core/mppi_common.cu rolloutKernel / normExpKernel / weightedReductionKernel,
gaussian.cu setGaussianControls, the Cartpole and Autorally plugins), compiled for sm_100 by oracle/ref_build/build.sh
with an Eigen stand-in ("reference kernels, shimmed host"), computed on a B200 for these workloads. Both sides seed
XORWOW with 42 and burn the one draw VanillaMPPI's constructor makes (mppi_controller.cu:95), so they consume the SAME
noise: per-sample trajectory costs must agree to the reference's own GPU-vs-CPU bar (1e-4 rel,
tests/mppi_core/rollout_kernel_tests.cu:258) and the optimal control / baseline / normaliser of a whole computeControl to
float accumulation differences. This turns "bit-exact sample indexing vs the reference kernels" from an argument into a test.
"""
import numpy as np
import pytest

from mppi_generic_b200 import host as H
from tests.golden import make_reference_gpu as G

pytestmark = pytest.mark.gpu
SEED = G.SEED


def _ours(w):
    """Our controller mirror: seeds XORWOW with SEED and burns the one draw VanillaMPPI's constructor makes."""
    return H.VanillaMPPIController(w.dyn, w.cost, None, w.sampler, w.dt, 1, w.lambda_, w.alpha, w.T, w.N, seed=SEED)


def _reference(stem, w):
    """The stored reference outputs, after checking that the workload builder still makes the inputs they came from."""
    g = G.load(stem)
    np.testing.assert_array_equal(w.x0, g["x0"])
    if "nn_theta" in g:
        np.testing.assert_array_equal(w.dyn.nn_theta, g["nn_theta"])
    return g


def _compare_costs(c_ref, ctl, w):
    ctl.engine.solve(w.x0, w.U0)  # one draw + K1 (+ K2) on the same generator position
    c = ctl.engine.get_costs()[0]
    return np.abs(c - c_ref) / np.maximum(np.abs(c_ref), 1.0)


@pytest.mark.parametrize("block", G.CARTPOLE_BLOCKS)
def test_cartpole_costs_and_solve_match_reference_gpu(block):
    w = G.cartpole_workload()
    ref = _reference(G.block_stem(block), w)
    ctl = _ours(w)
    for it in range(2):  # two consecutive draws: the generator offsets stay in step
        rel = _compare_costs(ref["costs"][it], ctl, w)
        assert rel.max() < 1e-4, (it, block, str(ref["kernel"]), rel.max(), int(rel.argmax()))
    ctl.computeControl(w.x0[0], 1)
    assert ctl.getBaselineCost() == pytest.approx(float(ref["baseline"]), rel=1e-5)
    assert ctl.getNormalizerCost() == pytest.approx(float(ref["normalizer"]), rel=1e-4)
    np.testing.assert_allclose(ctl.getControlSeq(), ref["U"], atol=1e-3)  # control range +-5, sigma 5


def test_both_reference_kernels_agree_with_ours():
    """The reference picks its single or its split rollout kernel by timing; the stored costs force each."""
    w = G.cartpole_workload()
    for split in (False, True):
        ref = _reference(G.kernel_stem(split), w)
        ctl = _ours(w)
        rel = _compare_costs(ref["costs"][0], ctl, w)
        # the split kernels' own bar against the CPU is 1e-3 (rollout_kernel_tests.cu:263-375)
        assert rel.max() < (1e-3 if split else 1e-4), (split, rel.max())


def test_autorally_costs_and_solve_match_reference_gpu():
    w = G.autorally_workload()
    ref = _reference(G.AUTORALLY_STEM, w)
    ctl = _ours(w)
    rel = _compare_costs(ref["costs"][0], ctl, w)
    # FP32 network evaluated two ways (the reference's FMA chains, our split tensor-core products) over a 100-step recurrence,
    # plus 1-texel map lookups: a sample whose wheel sits on a texel edge can land on the other side
    assert np.median(rel) < 2e-6, np.median(rel)
    assert np.quantile(rel, 0.99) < 1e-4, np.quantile(rel, 0.99)
    assert rel.max() < 5e-3, (rel.max(), int(rel.argmax()))
    ctl.computeControl(w.x0[0], 1)
    assert ctl.getBaselineCost() == pytest.approx(float(ref["baseline"]), rel=1e-4)
    assert ctl.getNormalizerCost() == pytest.approx(float(ref["normalizer"]), rel=2e-3)
    np.testing.assert_allclose(ctl.getControlSeq(), ref["U"], atol=2e-3)
