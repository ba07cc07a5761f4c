"""Python host for the b200 kernel set: a ctypes binding of ``include/neutral_b200.h`` and a
:class:`Simulation` that drives it the way the reference's C driver does
(``main.c:62-72`` initialise, ``main.c:85-147`` timestep loop, ``main.c:154-156`` validate).

The compute path is ``libneutral_b200.so`` only. There is no CPU fallback here: loading
fails loudly when the library has not been built, and every compute call fails loudly when
no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from .bank import F64_FIELDS, I32_FIELDS, HostBank, ParticleSoA, PARTICLE_AOS
from .build import LIB, build_library
from .decks import Problem, shard_range

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_u64p = C.POINTER(C.c_uint64)
_soa_p = C.POINTER(ParticleSoA)


class CrossSection(C.Structure):
    """ctypes mirror of the reference's ``CrossSection`` (``neutral_data.h:38-43``)."""

    _fields_ = [("keys", C.c_void_p), ("values", C.c_void_p), ("nentries", C.c_int)]


class NeutralB200Error(RuntimeError):
    pass


#: every symbol include/neutral_b200.h declares (checked by tests/test_cabi.py)
EXPORTED_SYMBOLS = [
    "solve_transport_2d", "inject_particles", "validate",
    "allocate_data", "allocate_float_data", "allocate_int_data", "allocate_uint64_data",
    "allocate_host_data", "allocate_host_float_data", "deallocate_data",
    "deallocate_host_data", "copy_buffer", "move_host_buffer_to_device", "initialise_devices",
    "nb200_solve_transport_2d_host",
    "nb200_abi_version", "nb200_last_error", "nb200_device_count", "nb200_set_stream",
    "nb200_set_shard", "nb200_bank_create", "nb200_bank_download", "nb200_bank_export",
    "nb200_bank_upload", "nb200_accumulate", "nb200_accumulate_clear", "nb200_accumulate_clear_async", "nb200_bank_copy", "nb200_bank_size", "nb200_bank_free", "nb200_memcpy_h2d",
    "nb200_memcpy_d2h", "nb200_memcpy_h2d_async", "nb200_memcpy_d2h_async", "nb200_bank_view",
    "nb200_bank_import", "nb200_memset_d", "nb200_synchronize", "nb200_set_option",
    "nb200_solve_finish", "nb200_last_step_stats", "nb200_kernel_launches", "nb200_selftest_rng_log",
    "nb200_selftest_log", "nb200_selftest_div", "nb200_selftest_fastmath", "nb200_selftest_cs", "nb200_host_threefry2x64_20",
    "nb200_host_log", "nb200_selftest_sincos", "nb200_host_sin", "nb200_host_cos",
    "nb200_selftest_dispatch_group",
    "nb200_host_sincos", "nb200_selftest_host_sincos",
    "nb200_bank_capacity", "nb200_bank_gpus", "nb200_bank_append", "nb200_get_option",
    "nb200_bank_set_option", "nb200_bank_solve_finish", "nb200_bank_pending", "nb200_mp_init",
    "nb200_mp_connect", "nb200_mp_finalize", "nb200_tally_sync", "nb200_update_replicas",
    "nb200_microbench_red", "nb200_bank_tally_batches", "nb200_bank_tally_relerr",
    "nb200_selftest_batch_of", "nb200_bank_set_flux_tally", "nb200_bank_set_batched_flux_tally",
    "nb200_bank_flux_batches", "nb200_bank_flux_relerr",
]

#: include/neutral_b200.h
NB200_BAD_OPTION = -2**31
NB200_MP_BLOB_BYTES = 256

_SOLVE_ARGS = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int,
               C.c_double, C.c_int, _ip, _ip, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
               C.c_void_p, C.c_void_p, C.POINTER(CrossSection), C.POINTER(CrossSection),
               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _u64p, _u64p]

_lib = None


def load_library(build: bool = False) -> C.CDLL:
    """Loads libneutral_b200.so. ``build=True`` (re)compiles it first when stale."""
    global _lib
    if _lib is not None:
        return _lib
    if build:
        build_library()
    if not os.path.exists(LIB):
        raise NeutralB200Error(
            f"{LIB} is missing: build it with `python -m neutral_b200.build` "
            "(the b200 kernel set has no CPU fallback)")
    L = C.CDLL(LIB)
    L.solve_transport_2d.argtypes = _SOLVE_ARGS
    L.solve_transport_2d.restype = None
    L.nb200_solve_transport_2d_host.argtypes = _SOLVE_ARGS
    L.nb200_solve_transport_2d_host.restype = None
    L.inject_particles.argtypes = [C.c_int] * 5 + [C.c_double] * 4 + [C.c_int, C.c_int,
                                  C.c_double, C.c_void_p, C.c_void_p, C.c_double,
                                  C.POINTER(_soa_p)]
    L.inject_particles.restype = C.c_size_t
    L.validate.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_void_p]
    L.validate.restype = None
    for name, ty in (("allocate_data", _dp), ("allocate_int_data", _ip),
                     ("allocate_uint64_data", _u64p)):
        f = getattr(L, name)
        f.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
        f.restype = C.c_size_t
    L.deallocate_data.argtypes = [C.c_void_p]
    L.initialise_devices.argtypes = [C.c_int]
    L.nb200_last_error.restype = C.c_char_p
    L.nb200_set_stream.argtypes = [C.c_void_p]
    L.nb200_set_shard.argtypes = [C.c_int, C.c_int]
    L.nb200_bank_create.argtypes = [_soa_p, C.c_int, C.c_int, C.POINTER(_soa_p)]
    L.nb200_bank_download.argtypes = [_soa_p, _soa_p]
    L.nb200_bank_export.argtypes = [_soa_p]
    L.nb200_bank_upload.argtypes = [_soa_p, _soa_p]
    L.nb200_accumulate.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.nb200_accumulate_clear.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.nb200_accumulate_clear_async.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.nb200_bank_copy.argtypes = [_soa_p, _soa_p]
    L.nb200_bank_size.argtypes = [_soa_p]
    L.nb200_bank_free.argtypes = [_soa_p]
    L.nb200_memcpy_h2d.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.nb200_memcpy_d2h.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.nb200_memcpy_h2d_async.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.nb200_memcpy_d2h_async.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.nb200_bank_view.argtypes = [_soa_p, _soa_p]
    L.nb200_bank_import.argtypes = [_soa_p]
    L.nb200_memset_d.argtypes = [C.c_void_p, C.c_int, C.c_size_t]
    L.nb200_set_option.argtypes = [C.c_char_p, C.c_int]
    L.nb200_get_option.argtypes = [C.c_char_p]
    L.nb200_bank_set_option.argtypes = [_soa_p, C.c_char_p, C.c_int]
    L.nb200_bank_solve_finish.argtypes = [_soa_p, _u64p, _u64p]
    L.nb200_bank_pending.argtypes = [_soa_p]
    L.nb200_bank_capacity.argtypes = [_soa_p]
    L.nb200_bank_gpus.argtypes = [_soa_p]
    L.nb200_bank_append.argtypes = [_soa_p, _soa_p, C.c_int]
    L.nb200_mp_init.argtypes = [C.c_int, C.c_int, C.c_size_t, C.c_void_p]
    L.nb200_mp_connect.argtypes = [C.c_void_p]
    L.nb200_tally_sync.argtypes = [C.c_void_p]
    L.nb200_microbench_red.argtypes = [C.c_int, C.c_size_t, C.c_int, _dp]
    L.nb200_bank_tally_batches.argtypes = [_soa_p, C.c_void_p, C.c_size_t]
    L.nb200_bank_tally_relerr.argtypes = [_soa_p, C.c_void_p, _dp]
    L.nb200_selftest_batch_of.argtypes = [C.c_uint64, C.c_uint64, C.c_int]
    L.nb200_selftest_batch_of.restype = C.c_uint
    L.nb200_bank_set_flux_tally.argtypes = [_soa_p, C.c_void_p, C.c_size_t]
    L.nb200_bank_set_batched_flux_tally.argtypes = [_soa_p, C.c_void_p, C.c_size_t]
    L.nb200_bank_flux_batches.argtypes = [_soa_p, C.c_void_p, C.c_size_t]
    L.nb200_bank_flux_relerr.argtypes = [_soa_p, C.c_void_p, _dp]
    L.nb200_last_step_stats.argtypes = [_u64p]
    L.nb200_solve_finish.argtypes = [_u64p, _u64p]
    L.nb200_kernel_launches.restype = C.c_uint64
    L.nb200_selftest_rng_log.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, _u64p,
                                         _dp, _dp]
    L.nb200_selftest_log.argtypes = [_dp, _dp, C.c_int]
    L.nb200_selftest_div.argtypes = [_dp, _dp, C.c_int, _dp, _dp]
    L.nb200_selftest_fastmath.argtypes = [_dp, _dp, C.c_int, _dp]
    L.nb200_selftest_cs.argtypes = [_dp, _dp, C.c_int, _dp, C.c_int, _ip, _dp]
    L.nb200_host_threefry2x64_20.argtypes = [C.c_uint64] * 4 + [_u64p]
    L.nb200_host_log.argtypes = [C.c_double]
    L.nb200_host_log.restype = C.c_double
    L.nb200_selftest_sincos.argtypes = [_dp, _dp, _dp, C.c_int]
    for name in ("nb200_host_sin", "nb200_host_cos"):
        getattr(L, name).argtypes = [C.c_double]
        getattr(L, name).restype = C.c_double
    L.nb200_host_sincos.argtypes = [_dp, C.c_longlong, _dp, _dp]
    L.nb200_host_sincos.restype = None
    L.nb200_selftest_host_sincos.argtypes = [_dp, C.c_longlong, _dp]
    L.nb200_selftest_host_sincos.restype = C.c_longlong
    _lib = L
    return L


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise NeutralB200Error(f"{what}: {load_library().nb200_last_error().decode()}")


def require_device() -> None:
    if load_library().nb200_device_count() <= 0:
        raise NeutralB200Error("no CUDA device available: the b200 kernel set has no CPU "
                               "fallback")


class DeviceArray:
    """A zero-filled device buffer from the kernel set's allocation layer."""

    _ALLOC = {np.dtype(np.float64): "allocate_data", np.dtype(np.int32): "allocate_int_data",
              np.dtype(np.uint64): "allocate_uint64_data"}

    def __init__(self, n: int, dtype=np.float64):
        self.lib = load_library()
        self.n = int(n)
        self.dtype = np.dtype(dtype)
        p = C.c_void_p()
        getattr(self.lib, self._ALLOC[self.dtype])(C.byref(p), self.n)
        self.ptr = p.value

    @classmethod
    def from_host(cls, a: np.ndarray) -> "DeviceArray":
        a = np.ascontiguousarray(a)
        d = cls(a.size, a.dtype)
        d.upload(a)
        return d

    @property
    def nbytes(self) -> int:
        return self.n * self.dtype.itemsize

    def upload(self, a: np.ndarray) -> None:
        a = np.ascontiguousarray(a, dtype=self.dtype)
        assert a.size == self.n
        _check(self.lib.nb200_memcpy_h2d(self.ptr, a.ctypes.data, self.nbytes), "memcpy_h2d")

    def download(self) -> np.ndarray:
        out = np.empty(self.n, dtype=self.dtype)
        _check(self.lib.nb200_memcpy_d2h(out.ctypes.data, self.ptr, self.nbytes), "memcpy_d2h")
        return out

    def zero(self) -> None:
        _check(self.lib.nb200_memset_d(self.ptr, 0, self.nbytes), "memset_d")

    def free(self) -> None:
        if self.ptr:
            self.lib.deallocate_data(self.ptr)
            self.ptr = None


@dataclass
class StepResult:
    facets: int
    collisions: int
    processed: int
    census: int
    deaths: int
    launches: int
    kernel_ns: int = 0
    sort_ns: int = 0

    @property
    def events(self) -> int:
        """Particle events of the step: facets + collisions + census (SURVEY.md 8d)."""
        return self.facets + self.collisions + self.census


class Simulation:
    """One problem resident on one GPU, stepped through ``solve_transport_2d``.

    ``rank``/``nranks`` select this GPU's contiguous particle shard (global RNG keys); the
    tally a step writes into can be redirected (``tally_ptr``) so that a multi-GPU host can
    all-reduce per-step deltas.
    """

    def __init__(self, problem: Problem, rank: int = 0, nranks: int = 1,
                 per_particle_counters: bool = True, quiet: bool = True, ngpus: int = 1,
                 tally_batches: int = 0, flux_tally: bool = False):
        self.lib = load_library()
        require_device()
        self.problem = problem
        d = problem.deck
        self.pid0, self.count = shard_range(d.nparticles, rank, nranks)
        self.rank, self.nranks = rank, nranks
        #: GPUs of THIS process the bank is sharded over (option "ngpus"): the library drives
        #: them all behind the same solve_transport_2d call and combines the tally itself
        self.ngpus = ngpus
        #: batches of the tally statistics (option "tally_batches", 0: none): the bank's
        #: deposits are kept per contiguous particle range, see :meth:`tally_relative_error`
        self.tally_batches = tally_batches
        if quiet:
            self.lib.nb200_set_option(b"print", 0)
        self.density = DeviceArray.from_host(problem.density.ravel())
        self.edgex = DeviceArray.from_host(problem.edgex)
        self.edgey = DeviceArray.from_host(problem.edgey)
        self.cs = []
        self._cs_arrays = []
        for keys, values in (problem.cs_scatter, problem.cs_absorb):
            dk, dv = DeviceArray.from_host(keys), DeviceArray.from_host(values)
            self._cs_arrays += [dk, dv]
            self.cs.append(CrossSection(dk.ptr, dv.ptr, len(keys)))
        self.tally = DeviceArray(d.nx * d.ny, np.float64)
        #: track-length flux per source particle (nb200_bank_set_flux_tally), attached to every
        #: bank this simulation creates; see :meth:`scalar_flux`. With ``tally_batches`` it is
        #: batched too (nb200_bank_set_batched_flux_tally), see :meth:`flux_relative_error`
        self.flux = DeviceArray(d.nx * d.ny, np.float64) if flux_tally else None
        self.counters = [DeviceArray(max(self.count, 1), np.uint64) for _ in range(3)] \
            if per_particle_counters else None
        self.bank = None
        self.bank_bytes = 0
        self.h2d_bytes = sum(a.nbytes for a in
                             [self.density, self.edgex, self.edgey] + self._cs_arrays)

    # -- bank ---------------------------------------------------------------------------
    def inject(self) -> int:
        """``inject_particles`` with the arguments ``neutral_data.c:109-114`` passes."""
        d, s = self.problem.deck, self.problem.source
        if self.bank is not None:
            self.lib.nb200_bank_free(self.bank)
        self.lib.nb200_set_shard(self.pid0, self.count if self.nranks > 1 else -1)
        prev = self._set_creation_options()
        out = _soa_p()
        self.bank_bytes = self.lib.inject_particles(
            d.nparticles, d.nx, d.nx, d.ny, 0, s.left, s.bottom, s.width, s.height, 0, 0,
            d.dt, self.edgex.ptr, self.edgey.ptr, d.initial_energy, C.byref(out))
        self._restore_options(prev)
        self.lib.nb200_set_shard(0, -1)
        self.bank = out
        self._attach_flux()
        return self.bank_bytes

    def load_bank(self, host: HostBank) -> None:
        """Uploads a host bank holding this shard's particles (injection order)."""
        assert len(host) == self.count
        if self.bank is not None:
            self.lib.nb200_bank_free(self.bank)
        st = host.as_struct()
        out = _soa_p()
        prev = self._set_creation_options()
        try:
            _check(self.lib.nb200_bank_create(C.byref(st), self.count, self.pid0, C.byref(out)),
                   "bank_create")
        finally:
            self._restore_options(prev)
        self.bank = out
        self._attach_flux()

    def _attach_flux(self) -> None:
        if self.flux is None:
            return
        if self.tally_batches:
            _check(self.lib.nb200_bank_set_batched_flux_tally(self.bank, self.flux.ptr,
                                                              self.flux.n),
                   "bank_set_batched_flux_tally")
        else:
            _check(self.lib.nb200_bank_set_flux_tally(self.bank, self.flux.ptr, self.flux.n),
                   "bank_set_flux_tally")

    def _set_creation_options(self) -> dict:
        prev = {}
        for name, value in ((b"ngpus", self.ngpus), (b"tally_batches", self.tally_batches)):
            prev[name] = self.lib.nb200_set_option(name, value)
            if prev[name] == NB200_BAD_OPTION:
                raise NeutralB200Error(f"option {name.decode()}={value}: "
                                       f"{self.lib.nb200_last_error().decode()}")
        return prev

    def _restore_options(self, prev: dict) -> None:
        for name, value in prev.items():
            if value != NB200_BAD_OPTION:
                self.lib.nb200_set_option(name, value)

    def bank_to_host(self) -> HostBank:
        host = HostBank.empty(self.count)
        st = host.as_struct()
        _check(self.lib.nb200_bank_download(self.bank, C.byref(st)), "bank_download")
        return host

    # -- stepping -----------------------------------------------------------------------
    def step(self, tt: int, tally_ptr: Optional[int] = None, defer: bool = False
             ) -> Optional[StepResult]:
        """One call of ``solve_transport_2d`` with ``master_key = tt`` (``main.c:101-110``).
        ``defer=True`` returns as soon as the timestep is enqueued (library option
        ``defer_finish``); :meth:`step_finish` then waits for it and returns the counts."""
        d = self.problem.deck
        self.lib.nb200_bank_set_option(self.bank, b"defer_finish", 1 if defer else 0)
        nlocal = C.c_int(self.count)
        facets, colls = C.c_uint64(0), C.c_uint64(0)
        ctr = [c.ptr for c in self.counters] if self.counters else [None] * 3
        self.lib.solve_transport_2d(
            d.nx, d.ny, d.nx, d.ny, tt, 0, 0, 0, d.dt, d.nparticles, C.byref(nlocal), None,
            C.cast(self.bank, C.c_void_p), self.density.ptr, self.edgex.ptr, self.edgey.ptr,
            None, None, C.byref(self.cs[0]), C.byref(self.cs[1]),
            tally_ptr if tally_ptr is not None else self.tally.ptr,
            ctr[0], ctr[1], ctr[2], C.byref(facets), C.byref(colls))
        if defer:
            return None
        return self._result(facets.value, colls.value)

    def step_finish(self) -> StepResult:
        """Completes a ``step(..., defer=True)``: waits for the timestep and returns its counts."""
        facets, colls = C.c_uint64(0), C.c_uint64(0)
        _check(self.lib.nb200_bank_solve_finish(self.bank, C.byref(facets), C.byref(colls)),
               "solve_finish")
        return self._result(facets.value, colls.value)

    def _result(self, facets: int, colls: int) -> StepResult:
        stats = (C.c_uint64 * 8)()
        self.lib.nb200_last_step_stats(stats)
        assert stats[0] == facets and stats[1] == colls
        return StepResult(int(stats[0]), int(stats[1]), int(stats[2]), int(stats[3]),
                          int(stats[4]), int(stats[5]), int(stats[6]), int(stats[7]))

    def run(self, iterations: Optional[int] = None) -> List[StepResult]:
        n = self.problem.deck.iterations if iterations is None else iterations
        return [self.step(tt) for tt in range(1, n + 1)]

    def run_pipelined(self, iterations: Optional[int] = None, first_tt: int = 1,
                      depth: int = 3, once_fed=None) -> List[StepResult]:
        """The same timesteps without a host round trip between them: up to ``depth`` steps
        are enqueued (``defer_finish``) before the oldest is collected, so the GPU goes from
        one timestep's history kernel straight into the next one's sort. Results are those of
        :meth:`run` (the steps execute in stream order either way). ``once_fed`` (optional
        callable) runs once, as soon as the GPU has ``depth`` timesteps queued: the place for
        host work that should not sit between two deck runs (enqueueing copies of other
        working sets)."""
        n = self.problem.deck.iterations if iterations is None else iterations
        out: List[StepResult] = []
        inflight = 0
        for tt in range(first_tt, first_tt + n):
            self.step(tt, defer=True)
            inflight += 1
            if once_fed is not None and (inflight >= depth or tt == first_tt + n - 1):
                once_fed()
                once_fed = None
            if inflight >= depth:
                out.append(self.step_finish())
                inflight -= 1
        while inflight:
            out.append(self.step_finish())
            inflight -= 1
        self.lib.nb200_bank_set_option(self.bank, b"defer_finish", 0)
        return out

    def tally_sync(self) -> None:
        """Brings ``self.tally`` up to date in a sharded run (a collective in a multi-process
        group: every rank calls it)."""
        _check(self.lib.nb200_tally_sync(self.tally.ptr), "tally_sync")

    # -- results ------------------------------------------------------------------------
    def tally_to_host(self) -> np.ndarray:
        return self.tally.download()

    def tally_batches_to_host(self) -> np.ndarray:
        """(B, ny, nx) cumulative partial tallies of the B particle batches (option
        ``tally_batches``); flushes the caller's tally first."""
        d = self.problem.deck
        ncells = d.nx * d.ny
        out = DeviceArray(self.tally_batches * ncells, np.float64)
        try:
            rc = self.lib.nb200_bank_tally_batches(self.bank, out.ptr, ncells)
            if rc != self.tally_batches:
                raise NeutralB200Error(
                    f"bank_tally_batches: {self.lib.nb200_last_error().decode()}")
            return out.download().reshape(self.tally_batches, d.ny, d.nx)
        finally:
            out.free()

    def tally_relative_error(self) -> Tuple[np.ndarray, float]:
        """Relative error of the tally from its batches: (R per cell as (ny, nx), R of the
        tally total). R = sqrt(s^2 / B) / |m| over the batch estimates x_b = S_b N / n_b."""
        d = self.problem.deck
        out = DeviceArray(d.nx * d.ny, np.float64)
        total = C.c_double(0.0)
        try:
            _check(self.lib.nb200_bank_tally_relerr(self.bank, out.ptr, C.byref(total)),
                   "bank_tally_relerr")
            return out.download().reshape(d.ny, d.nx), float(total.value)
        finally:
            out.free()

    def flux_to_host(self) -> np.ndarray:
        """(ny, nx) track length per source particle in every cell, summed over timesteps
        (``flux_tally=True``)."""
        d = self.problem.deck
        return self.flux.download().reshape(d.ny, d.nx)

    def scalar_flux(self) -> np.ndarray:
        """(ny, nx) time-integrated scalar flux per source particle: :meth:`flux_to_host`
        divided by the cell areas dx_i dy_j."""
        dx = np.diff(self.problem.edgex)
        dy = np.diff(self.problem.edgey)
        return self.flux_to_host() / np.outer(dy, dx)

    def flux_batches_to_host(self) -> np.ndarray:
        """(B, ny, nx) cumulative partial fluxes of the B particle batches (``flux_tally=True``
        with ``tally_batches``); flushes the flux array first."""
        d = self.problem.deck
        ncells = d.nx * d.ny
        out = DeviceArray(self.tally_batches * ncells, np.float64)
        try:
            rc = self.lib.nb200_bank_flux_batches(self.bank, out.ptr, ncells)
            if rc != self.tally_batches:
                raise NeutralB200Error(
                    f"bank_flux_batches: {self.lib.nb200_last_error().decode()}")
            return out.download().reshape(self.tally_batches, d.ny, d.nx)
        finally:
            out.free()

    def flux_relative_error(self) -> Tuple[np.ndarray, float]:
        """Relative error of the flux from its batches: (R per cell as (ny, nx), R of the flux
        total), with the estimator of :meth:`tally_relative_error`. :meth:`scalar_flux` has the
        same R per cell, because it divides every batch of a cell by the same exact constant,
        the cell's area."""
        d = self.problem.deck
        out = DeviceArray(d.nx * d.ny, np.float64)
        total = C.c_double(0.0)
        try:
            _check(self.lib.nb200_bank_flux_relerr(self.bank, out.ptr, C.byref(total)),
                   "bank_flux_relerr")
            return out.download().reshape(d.ny, d.nx), float(total.value)
        finally:
            out.free()

    def counters_to_host(self) -> np.ndarray:
        """(3, count) cumulative per-particle facets / collisions / census events."""
        return np.stack([c.download()[: self.count] for c in self.counters])

    def validate(self, params_filename: Optional[str] = None) -> None:
        d = self.problem.deck
        name = (params_filename or d.path).encode()
        self.lib.validate(d.nx, d.ny, name, 0, self.tally.ptr)

    def free(self) -> None:
        if self.bank is not None:
            self.lib.nb200_bank_free(self.bank)
            self.bank = None
        for a in [self.density, self.edgex, self.edgey, self.tally] + self._cs_arrays + \
                (self.counters or []) + ([self.flux] if self.flux is not None else []):
            a.free()


def solve_transport_2d_host(problem: Problem, aos: np.ndarray, master_key: int,
                            tally: np.ndarray, counters: Optional[np.ndarray] = None
                            ) -> Tuple[int, int]:
    """The host-buffer flavour (``nb200_solve_transport_2d_host``): omp3's signature on host
    arrays. ``aos`` (:data:`PARTICLE_AOS`) and ``tally`` are updated in place; returns
    (facets, collisions)."""
    lib = load_library()
    require_device()
    d = problem.deck
    assert aos.dtype == PARTICLE_AOS and aos.flags["C_CONTIGUOUS"]
    assert tally.dtype == np.float64 and tally.size == d.nx * d.ny
    (sk, sv), (ak, av) = problem.cs_scatter, problem.cs_absorb
    cs_s = CrossSection(sk.ctypes.data, sv.ctypes.data, len(sk))
    cs_a = CrossSection(ak.ctypes.data, av.ctypes.data, len(ak))
    nlocal = C.c_int(len(aos))
    facets, colls = C.c_uint64(0), C.c_uint64(0)
    ctr = [counters[i].ctypes.data for i in range(3)] if counters is not None else [None] * 3
    lib.nb200_solve_transport_2d_host(
        d.nx, d.ny, d.nx, d.ny, master_key, 0, 0, 0, d.dt, d.nparticles, C.byref(nlocal),
        None, aos.ctypes.data, problem.density.ctypes.data, problem.edgex.ctypes.data,
        problem.edgey.ctypes.data, None, None, C.byref(cs_s), C.byref(cs_a),
        tally.ctypes.data, ctr[0], ctr[1], ctr[2], C.byref(facets), C.byref(colls))
    return int(facets.value), int(colls.value)
