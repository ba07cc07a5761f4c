"""The reference of the track-length flux tally (TEST INFRASTRUCTURE): ``tests/flux_reference.c``,
the oracle port's timestep plus a flux output, compiled with the oracle port's flags into a
temporary directory (the tree may be read-only) once per process.

:func:`flux_reference` returns an object whose ``step`` takes the arguments of
``oracle.oracle.OraclePort.step`` plus ``flux`` (nx * ny float64, accumulated in place, or None).
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
from typing import Optional

import numpy as np

from neutral_b200.bank import ParticleSoA

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCE = os.path.join(HERE, "flux_reference.c")
# oracle/Makefile, target `port`
CFLAGS = ["-O2", "-std=gnu99", "-fopenmp", "-march=x86-64-v3", "-ffp-contract=off", "-Wall",
          "-fPIC", "-shared"]

_dp = C.POINTER(C.c_double)
_u64p = C.POINTER(C.c_uint64)


def _ptr(a: np.ndarray, ty=_dp):
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(ty)


class FluxReference:
    def __init__(self):
        tmp = tempfile.mkdtemp(prefix="nb200_flux_reference_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libflux_reference.so")
        subprocess.run(["gcc"] + CFLAGS + [SOURCE, "-o", so, "-lm"],
                       check=True)
        self.lib = C.CDLL(so)
        self.lib.flux_reference_transport_step.argtypes = [
            C.c_int, C.c_int, C.c_uint64, C.c_double, C.c_int, C.c_int, C.c_int,
            C.POINTER(ParticleSoA), _dp, _dp, _dp, _dp, _dp, C.c_int, _dp, _dp, C.c_int,
            _dp, _u64p, _u64p, _u64p, _u64p, _dp]

    def step(self, prob, bank, master_key: int, tally: np.ndarray, pid0: int = 0,
             counters=None, ntotal: Optional[int] = None, flux: Optional[np.ndarray] = None):
        """One timestep in place, as OraclePort.step; returns (facets, collisions, processed)."""
        d = prob.deck
        st = bank.as_struct()
        totals = (C.c_uint64 * 3)()
        if counters is not None:
            assert counters.shape == (3, len(bank)) and counters.dtype == np.uint64
            cf, cc, cz = (_ptr(counters[i], _u64p) for i in range(3))
        else:
            cf = cc = cz = None
        if flux is not None:
            assert flux.dtype == np.float64 and flux.size == d.nx * d.ny
        (sk, sv), (ak, av) = prob.cs_scatter, prob.cs_absorb
        self.lib.flux_reference_transport_step(
            d.nx, d.ny, master_key, d.dt, ntotal or d.nparticles, pid0, len(bank),
            C.byref(st), _ptr(prob.density), _ptr(prob.edgex), _ptr(prob.edgey),
            _ptr(sk), _ptr(sv), len(sk), _ptr(ak), _ptr(av), len(ak),
            _ptr(tally), cf, cc, cz, totals, None if flux is None else _ptr(flux))
        return int(totals[0]), int(totals[1]), int(totals[2])


_instance: Optional[FluxReference] = None


def flux_reference() -> FluxReference:
    global _instance
    if _instance is None:
        _instance = FluxReference()
    return _instance
