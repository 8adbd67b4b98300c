"""ctypes binding of oracle/_ref/libmppi_ref_gpu.so — the UNMODIFIED reference GPU path (VanillaMPPIController + the
reference's own kernels, built by oracle/ref_build/build.sh from the reference's sources with an Eigen stand-in:
"reference kernels, shimmed host"). TEST / BENCH INFRASTRUCTURE ONLY: imported by tests/golden/make_reference_gpu.py,
which stores what the reference computes for tests/test_gpu_vs_reference.py, and by bench.py's `reference_gpu` block;
never by the product package. The reference's sources are needed to build the library, not to run it.
"""
from __future__ import annotations

import ctypes as C
import os
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libmppi_ref_gpu.so")
_lib = None


def available() -> bool:
    return os.path.exists(LIB_PATH)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = C.CDLL(LIB_PATH)
        _lib.refgpu_last_error.restype = C.c_char_p
        _lib.refgpu_create_cartpole.restype = C.c_void_p
        _lib.refgpu_create_autorally.restype = C.c_void_p
        _lib.refgpu_time_compute_control.restype = C.c_double
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class RefController:
    """One reference VanillaMPPIController (a fixed <T, N> instantiation of the harness)."""

    def __init__(self, handle):
        if not handle:
            raise RuntimeError("reference controller: " + lib().refgpu_last_error().decode())
        self._h = C.c_void_p(handle)
        n, t, s, c = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        lib().refgpu_dims(self._h, C.byref(n), C.byref(t), C.byref(s), C.byref(c))
        self.N, self.T, self.S, self.C = n.value, t.value, s.value, c.value

    def close(self):
        if self._h:
            lib().refgpu_destroy(self._h)
            self._h = None

    def kernel_choice(self) -> str:
        return "split" if lib().refgpu_kernel_choice(self._h) else "single"

    def force_kernel(self, split: bool) -> None:
        lib().refgpu_force_kernel(self._h, int(split))

    def rollout_costs(self, x0, stride: int = 1) -> np.ndarray:
        """generateSamples + the reference rollout kernel(s); the per-sample costs before they become weights
        (mppi_controller.cu:155-186). Advances the generator like one computeControl."""
        costs = np.empty(self.N, np.float32)
        if lib().refgpu_rollout_costs(self._h, _p(_f32(x0)), stride, _p(costs)):
            raise RuntimeError(lib().refgpu_last_error().decode())
        return costs

    def compute_control(self, x0, stride: int = 1):
        U = np.empty((self.T, self.C), np.float32)
        st = np.empty(2, np.float32)
        if lib().refgpu_compute_control(self._h, _p(_f32(x0)), stride, _p(U), _p(st)):
            raise RuntimeError(lib().refgpu_last_error().decode())
        return U, float(st[0]), float(st[1])

    def set_control(self, U) -> None:
        lib().refgpu_set_control(self._h, _p(_f32(U)))

    def time_compute_control(self, x0, stride: int = 1, warmup: int = 10, iters: int = 100) -> float:
        """Seconds per computeControl, steady_clock around the host call (tests/controllers/vanilla_mppi_test.cu:290-292)."""
        return float(lib().refgpu_time_compute_control(self._h, _p(_f32(x0)), stride, warmup, iters))


def _blk(block):
    b = tuple(block) if len(block) == 4 else tuple(block) + tuple(block)
    return (C.c_int * 4)(*b)


def cartpole(w, seed: int, small: bool = False, block=(64, 4)) -> RefController:
    """The reference controller for a workloads.cartpole() description `w` (N must be 8192, or 2048 with small=True; T 100).
    block = (dynamics x, y) or (dynamics x, y, cost x, y): dynamics_rollout_dim_ / cost_rollout_dim_."""
    assert w.T == 100 and w.N == (2048 if small else 8192), (w.N, w.T)
    cp, lim, sp = w.cost.params, w.dyn.params.lim, w.sampler.params
    p = _f32([w.dyn.params.cart_mass, w.dyn.params.pole_mass, w.dyn.params.pole_length, lim.rng_lo[0], lim.rng_hi[0],
              cp.cart_position_coeff, cp.cart_velocity_coeff, cp.pole_angle_coeff, cp.pole_angular_velocity_coeff,
              cp.control_cost_coeff[0], cp.terminal_cost_coeff, *list(cp.desired_terminal_state)[:4],
              sp.std_dev[0], sp.control_cost_coeff[0], sp.pure_noise_trajectories_percentage, w.dt, w.lambda_, w.alpha])
    return RefController(lib().refgpu_create_cartpole(1 if small else 0, _p(p), C.c_uint(seed), _blk(block)))


def write_track_npz(path: str, ch0: np.ndarray, xb, yb, ppm: float) -> None:
    """The npz layout ARStandardCost::loadTrackData reads (ar_standard_cost.cu:85-142; scripts/autorally/test/generateTestMaps.py)."""
    z = np.zeros_like(ch0, dtype=np.float32)
    np.savez(path, xBounds=_f32(xb), yBounds=_f32(yb), pixelsPerMeter=_f32([ppm]), channel0=_f32(ch0).ravel(),
             channel1=z.ravel(), channel2=z.ravel(), channel3=z.ravel())


def autorally(w, seed: int, small: bool = False, block=(64, 8)) -> RefController:
    """The reference controller for a workloads.autorally() description `w` (N must be 32768, or 4096 with small=True; T 100).
    The synthetic track map goes through the reference's own loadTrackData (npz via its vendored cnpy)."""
    from mppi_generic_b200 import workloads as W
    assert w.T == 100 and w.N == (4096 if small else 32768), (w.N, w.T)
    lim, sp = w.dyn.params.lim, w.sampler.params
    ch0, xb, yb, ppm = W.track_map_standard()
    d = tempfile.mkdtemp(prefix="refgpu_")
    path = os.path.join(d, "track_map_standard.npz")
    write_track_npz(path, ch0, xb, yb, ppm)
    theta = _f32(w.dyn.nn_theta)
    p = _f32([lim.rng_lo[0], lim.rng_hi[0], lim.rng_lo[1], lim.rng_hi[1], sp.std_dev[0], sp.std_dev[1],
              sp.control_cost_coeff[0], sp.control_cost_coeff[1], sp.pure_noise_trajectories_percentage,
              w.dt, w.lambda_, w.alpha])
    h = lib().refgpu_create_autorally(1 if small else 0, _p(theta), theta.size, path.encode(), _p(p), C.c_uint(seed),
                                      _blk(block))
    return RefController(h)
