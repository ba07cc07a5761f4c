"""The reference of the energy-group flux tally (TEST INFRASTRUCTURE):
``tests/group_flux_reference.c``, the oracle port's timestep with a group-resolved flux output,
compiled with the oracle port's flags into a temporary directory (the tree may be read-only) once
per process.

:func:`group_flux_reference` returns an object whose ``step`` takes the arguments of
``oracle.oracle.OraclePort.step`` plus ``gflux`` (G * nx * ny float64, group-major, accumulated in
place, or None) and ``edges`` (G + 1 float64).
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

from flux_reference import CFLAGS, _dp, _ptr, _u64p
from neutral_b200.bank import ParticleSoA

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCE = os.path.join(HERE, "group_flux_reference.c")


class GroupFluxReference:
    def __init__(self):
        tmp = tempfile.mkdtemp(prefix="nb200_group_flux_reference_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libgroup_flux_reference.so")
        subprocess.run(["gcc"] + CFLAGS + [SOURCE, "-o", so, "-lm"], check=True)
        self.lib = C.CDLL(so)
        self.lib.group_flux_reference_transport_step.argtypes = [
            C.c_int, C.c_int, C.c_uint64, C.c_double, C.c_int, C.c_int, C.c_int,
            C.POINTER(ParticleSoA), _dp, _dp, _dp, _dp, _dp, C.c_int, _dp, _dp, C.c_int,
            _dp, _u64p, _u64p, _u64p, _u64p, _dp, _dp, C.c_int]

    def step(self, prob, bank, master_key: int, tally: np.ndarray, pid0: int = 0,
             counters=None, ntotal: Optional[int] = None, gflux: Optional[np.ndarray] = None,
             edges: Optional[np.ndarray] = None):
        """One timestep in place, as OraclePort.step; returns (facets, collisions, processed)."""
        d = prob.deck
        st = bank.as_struct()
        totals = (C.c_uint64 * 3)()
        if counters is not None:
            assert counters.shape == (3, len(bank)) and counters.dtype == np.uint64
            cf, cc, cz = (_ptr(counters[i], _u64p) for i in range(3))
        else:
            cf = cc = cz = None
        ngroups = 0
        if gflux is not None:
            edges = np.ascontiguousarray(edges, dtype=np.float64)
            ngroups = edges.size - 1
            assert ngroups >= 1 and np.all(np.diff(edges) > 0)
            assert gflux.dtype == np.float64 and gflux.size == ngroups * d.nx * d.ny
        (sk, sv), (ak, av) = prob.cs_scatter, prob.cs_absorb
        self.lib.group_flux_reference_transport_step(
            d.nx, d.ny, master_key, d.dt, ntotal or d.nparticles, pid0, len(bank),
            C.byref(st), _ptr(prob.density), _ptr(prob.edgex), _ptr(prob.edgey),
            _ptr(sk), _ptr(sv), len(sk), _ptr(ak), _ptr(av), len(ak),
            _ptr(tally), cf, cc, cz, totals, None if gflux is None else _ptr(gflux),
            None if gflux is None else _ptr(edges), ngroups)
        return int(totals[0]), int(totals[1]), int(totals[2])


_instance: Optional[GroupFluxReference] = None


def group_flux_reference() -> GroupFluxReference:
    global _instance
    if _instance is None:
        _instance = GroupFluxReference()
    return _instance
