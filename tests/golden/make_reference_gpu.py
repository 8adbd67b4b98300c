"""Regenerates tests/golden/reference_gpu/: what the unmodified reference GPU path computed for the cases of
tests/test_gpu_vs_reference.py, so that the comparison runs without the reference's sources or its build.

Needs a CUDA device and oracle/_ref/libmppi_ref_gpu.so, which oracle/ref_build/build.sh compiles from the reference's own
VanillaMPPIController and kernels with an Eigen stand-in ("reference kernels, shimmed host"):

    python tests/golden/make_reference_gpu.py

Each .npz holds the initial state the workload builder made (the test checks it still does) and the reference's
outputs in the order the test consumes them: the per-sample rollout costs of consecutive noise draws, then, where the
test solves, one computeControl (optimal control sequence, baseline, normaliser) on the next draw.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from mppi_generic_b200 import workloads as W  # noqa: E402

SEED = 42
# block shapes the reference accepts: its cost block x must not exceed num_timesteps (mppi_common.cu:1274 exits otherwise)
CARTPOLE_BLOCKS = [(64, 4), (32, 1), (64, 2, 100, 1)]
AUTORALLY_STEM = "autorally_N4096_T100"


def cartpole_workload():
    return W.cartpole(2048, 100)


def autorally_workload():
    return W.autorally(4096, 100)


def block_stem(block) -> str:
    return "cartpole_N2048_T100_block" + "x".join(str(b) for b in block)


def kernel_stem(split: bool) -> str:
    return "cartpole_N2048_T100_" + ("split" if split else "single") + "_kernel"


def path(stem: str) -> str:
    return os.path.join(HERE, "reference_gpu", stem + ".npz")


def load(stem: str):
    return np.load(path(stem))


def main():
    from oracle import ref_gpu as RG
    os.makedirs(os.path.join(HERE, "reference_gpu"), exist_ok=True)
    w = cartpole_workload()
    for block in CARTPOLE_BLOCKS:
        ref = RG.cartpole(w, SEED, small=True, block=block)
        costs = [ref.rollout_costs(w.x0[0]) for _ in range(2)]
        kernel = ref.kernel_choice()
        U, baseline, normalizer = ref.compute_control(w.x0[0])
        ref.close()
        np.savez_compressed(path(block_stem(block)), x0=w.x0, costs=np.stack(costs), kernel=kernel, U=U, baseline=baseline,
                            normalizer=normalizer)
    for split in (False, True):
        ref = RG.cartpole(w, SEED, small=True)
        ref.force_kernel(split)
        costs = ref.rollout_costs(w.x0[0])
        ref.close()
        np.savez_compressed(path(kernel_stem(split)), x0=w.x0, costs=costs[None])
    w = autorally_workload()
    ref = RG.autorally(w, SEED, small=True)
    costs = ref.rollout_costs(w.x0[0])
    kernel = ref.kernel_choice()
    U, baseline, normalizer = ref.compute_control(w.x0[0])
    ref.close()
    np.savez_compressed(path(AUTORALLY_STEM), x0=w.x0, nn_theta=w.dyn.nn_theta, costs=costs[None], kernel=kernel, U=U,
                        baseline=baseline, normalizer=normalizer)
    for f in sorted(os.listdir(os.path.join(HERE, "reference_gpu"))):
        print(f, os.path.getsize(os.path.join(HERE, "reference_gpu", f)), "bytes")


if __name__ == "__main__":
    main()
