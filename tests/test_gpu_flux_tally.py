"""The track-length flux tally on the GPU (nb200_bank_set_flux_tally): attaching a flux array
changes no history and no energy deposit; the flux equals the reference's after every
timestep (the oracle port's timestep with a flux output, tests/flux_reference.c); it sums to the
distance travelled and reproduces chord lengths; detaching stops it;
and every refusal comes back as an error code or, at enqueue, a fatal error with its message."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import SMALL_DECKS
from neutral_b200.decks import build_problem
from neutral_b200.host import NB200_BAD_OPTION, DeviceArray, Simulation, _soa_p
from flux_reference import flux_reference
from test_flux_tally_cpu import (check_chords, check_stream, ray_bank, ray_problem,
                                 stream_expectations)
from test_gpu_parity import DEFAULTS, MODES, tally_close
from variants import VARIANTS

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _problem(name):
    return VARIANTS[name]() if name in VARIANTS else build_problem(name)


def _set_mode(lib, name):
    for k, v in MODES[name].items():
        assert lib.nb200_set_option(k.encode(), v) != NB200_BAD_OPTION


@pytest.fixture(params=["pipeline", "pipeline-ieee-div", "pipeline-class-only"])
def kernel_mode(request, gpu_lib):
    _set_mode(gpu_lib, request.param)
    yield request.param
    for k, v in DEFAULTS.items():
        gpu_lib.nb200_set_option(k.encode(), v)


def _run(prob, flux, pipelined=False, port=None):
    """Per-timestep counts, bank after every timestep (step by step) or at the end (pipelined),
    per-particle counters, the energy tally and the flux. With `port`, the flux after every
    timestep is checked against the flux reference run on the port's injected bank."""
    sim = Simulation(prob, flux_tally=flux)
    sim.inject()
    d = prob.deck
    counts, banks = [], []
    if port is not None:
        pbank = port.inject(prob)
        ptally, pflux = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
    if pipelined:
        counts = [(r.facets, r.collisions, r.processed, r.census, r.deaths)
                  for r in sim.run_pipelined(depth=3)]
        banks.append(sim.bank_to_host())
        if port is not None:
            for tt in range(1, d.iterations + 1):
                flux_reference().step(prob, pbank, tt, ptally, flux=pflux)
            assert tally_close(sim.flux_to_host().ravel(), pflux)
    else:
        for tt in range(1, d.iterations + 1):
            r = sim.step(tt)
            counts.append((r.facets, r.collisions, r.processed, r.census, r.deaths))
            banks.append(sim.bank_to_host())
            if port is not None:
                flux_reference().step(prob, pbank, tt, ptally, flux=pflux)
                assert tally_close(sim.flux_to_host().ravel(), pflux), tt
    out = dict(counts=counts, banks=banks, counters=sim.counters_to_host(),
               tally=sim.tally_to_host())
    if flux:
        out["flux"] = sim.flux_to_host()
    sim.free()
    return out


def _same_histories(got, want):
    assert got["counts"] == want["counts"]
    for tt, (a, b) in enumerate(zip(got["banks"], want["banks"])):
        diff = a.bit_equal(b)
        assert sum(diff.values()) == 0, (tt, diff)
    assert np.array_equal(got["counters"], want["counters"])
    assert tally_close(got["tally"], want["tally"])


@pytest.mark.parametrize("name", SMALL_DECKS + list(VARIANTS))
def test_histories_unchanged_and_flux_matches_the_port(gpu_lib, port, kernel_mode, name):
    """1 and 2: bit-identical histories and a 1e-10 energy tally with flux attached; the flux
    equals the reference's per cell (1e-10) after every timestep, step by step and pipelined."""
    prob = _problem(name)
    for pipelined in (False, True):
        base = _run(prob, False, pipelined)
        got = _run(prob, True, pipelined, port=port)
        _same_histories(got, base)
        assert np.count_nonzero(got["flux"]) > 0


@pytest.mark.parametrize("name", ["csp_small", "mixed_small"])
def test_without_the_step_graph(gpu_lib, port, name):
    """1 and 2 with the timestep's calls issued one by one (step_graph=0)."""
    _set_mode(gpu_lib, "pipeline-calls")
    try:
        prob = _problem(name)
        _same_histories(_run(prob, True, port=port), _run(prob, False))
    finally:
        for k, v in DEFAULTS.items():
            gpu_lib.nb200_set_option(k.encode(), v)


def test_stream_sums_to_the_distance_travelled(gpu_lib, port):
    """3, (b) on the device: every timestep's flux sums to v(E0) dt; energy = flux (sigma_t
    BARNS) response nd per cell."""
    prob = build_problem("stream_small")
    d = prob.deck
    want_sum, factor = stream_expectations(port, prob)
    sim = Simulation(prob, flux_tally=True)
    sim.inject()
    sums = []
    for tt in range(1, d.iterations + 1):
        before = sim.flux_to_host().sum()
        r = sim.step(tt)
        assert r.collisions == 0 and r.processed == d.nparticles
        sums.append(sim.flux_to_host().sum() - before)
    check_stream(sums, want_sum, sim.flux_to_host().ravel(), sim.tally_to_host(), factor)
    sim.free()


def test_chord_lengths(gpu_lib):
    """3, (c) on the device: one particle, per-cell flux = the ray march's chord lengths."""
    prob = ray_problem()
    sim = Simulation(prob, flux_tally=True)
    sim.load_bank(ray_bank(prob))
    for tt in range(1, prob.deck.iterations + 1):
        r = sim.step(tt)
        assert r.collisions == 0 and r.processed == 1
    check_chords(sim.flux_to_host().ravel(), prob)
    sim.free()


def test_full_csp_against_the_port(gpu_lib, port):
    """4: the full csp deck, flux per cell against the flux reference run on the host cores (1e-10)."""
    prob = build_problem("csp")
    d = prob.deck
    sim = Simulation(prob, per_particle_counters=False, flux_tally=True)
    sim.inject()
    sim.run_pipelined()
    got = sim.flux_to_host().ravel()
    sim.free()
    bank = port.inject(prob)
    tally, flux = np.zeros(d.nx * d.ny), np.zeros(d.nx * d.ny)
    for tt in range(1, d.iterations + 1):
        flux_reference().step(prob, bank, tt, tally, flux=flux)
    assert np.count_nonzero(flux) > 0
    assert tally_close(got, flux)


def _set_flux(lib, sim, arr):
    return lib.nb200_bank_set_flux_tally(sim.bank, arr.ptr if arr is not None else None,
                                         arr.n if arr is not None else 0)


def test_detach_reattach_and_two_banks(gpu_lib, port):
    """5: after detaching, further timesteps leave the array bitwise untouched and the bank
    continues bit-identical; a second array attached later receives exactly the later
    timesteps' flux; a bank with flux and one without, stepped alternately, are both right."""
    lib = gpu_lib
    prob = build_problem("csp_small", iterations=5)
    d = prob.deck
    base = _run(prob, False)
    pbank = port.inject(prob)
    ptally = np.zeros(d.nx * d.ny)
    pflux = [np.zeros(d.nx * d.ny) for _ in range(d.iterations)]
    for tt in range(1, d.iterations + 1):
        flux_reference().step(prob, pbank, tt, ptally, flux=pflux[tt - 1])

    sim = Simulation(prob, flux_tally=True)
    sim.inject()
    sim.step(1)
    assert tally_close(sim.flux_to_host().ravel(), pflux[0])
    assert _set_flux(lib, sim, None) == 0
    frozen = sim.flux_to_host().copy()
    second = DeviceArray(d.nx * d.ny)
    for tt in range(2, d.iterations + 1):
        if tt == 4:
            assert _set_flux(lib, sim, second) == 0
        sim.step(tt)
        assert np.array_equal(sim.flux_to_host().view(np.uint64), frozen.view(np.uint64)), tt
        assert sum(sim.bank_to_host().bit_equal(base["banks"][tt - 1]).values()) == 0, tt
    assert tally_close(second.download(), pflux[3] + pflux[4])
    assert tally_close(sim.tally_to_host(), base["tally"])
    sim.free()
    second.free()

    a = Simulation(prob, flux_tally=True)
    b = Simulation(prob)
    a.inject()
    b.inject()
    for tt in range(1, d.iterations + 1):
        ra, rb = a.step(tt), b.step(tt)
        assert (ra.facets, ra.collisions) == (rb.facets, rb.collisions) == base["counts"][tt - 1][:2]
        for s in (a, b):
            assert sum(s.bank_to_host().bit_equal(base["banks"][tt - 1]).values()) == 0, tt
    assert tally_close(a.flux_to_host().ravel(), sum(pflux))
    assert tally_close(a.tally_to_host(), base["tally"])
    assert tally_close(b.tally_to_host(), base["tally"])
    a.free()
    b.free()


def test_refusals(gpu_lib):
    """6: every refusal returns its code and says why."""
    lib = gpu_lib
    prob = build_problem("csp_small")
    n = prob.deck.nx * prob.deck.ny

    def refused(rc, word, code=-3):
        assert rc == code, (rc, word)
        assert word.encode() in lib.nb200_last_error(), lib.nb200_last_error()

    flux = DeviceArray(n)
    junk = (C.c_double * 4)()
    not_a_bank = C.cast(C.addressof(junk), _soa_p)
    refused(lib.nb200_bank_set_flux_tally(not_a_bank, flux.ptr, n), "not a bank handle")

    sim = Simulation(prob)
    sim.inject()
    sim.step(1, defer=True)
    refused(_set_flux(lib, sim, flux), "enqueued", code=-4)
    sim.step_finish()
    lib.nb200_bank_set_option(sim.bank, b"defer_finish", 0)
    host = np.zeros(n)
    refused(lib.nb200_bank_set_flux_tally(sim.bank, host.ctypes.data, n), "not device memory")
    refused(lib.nb200_bank_set_flux_tally(sim.bank, flux.ptr, 0), "cells")
    for name, value in ((b"pipeline", 0), (b"tally_prereduce", 1)):
        prev = lib.nb200_bank_set_option(sim.bank, name, value)
        refused(_set_flux(lib, sim, flux), "pipeline=1 and tally_prereduce=0")
        lib.nb200_bank_set_option(sim.bank, name, prev)
    assert _set_flux(lib, sim, flux) == 0
    assert lib.nb200_bank_set_option(sim.bank, b"pipeline", 0) == NB200_BAD_OPTION
    assert b"flux tally" in lib.nb200_last_error()
    assert lib.nb200_bank_set_option(sim.bank, b"tally_prereduce", 1) == NB200_BAD_OPTION
    assert lib.nb200_bank_set_option(sim.bank, b"fast_div", 0) != NB200_BAD_OPTION
    lib.nb200_bank_set_option(sim.bank, b"fast_div", 1)
    sim.free()

    batched = Simulation(prob, tally_batches=4)
    batched.inject()
    refused(_set_flux(lib, batched, flux), "tally_batches")
    batched.free()

    blob = (C.c_char * 256)()
    assert lib.nb200_mp_init(2, 0, n, blob) == 0
    try:
        grouped = Simulation(prob)
        grouped.inject()
        refused(_set_flux(lib, grouped, flux), "multi-process group")
        grouped.free()
    finally:
        lib.nb200_mp_finalize()
    flux.free()


def test_sharded_bank_is_refused(gpu_lib):
    if gpu_lib.nb200_device_count() < 2:
        pytest.skip("a bank sharded over several GPUs needs at least two")
    prob = build_problem("csp_small")
    sim = Simulation(prob, ngpus=2)
    sim.inject()
    flux = DeviceArray(prob.deck.nx * prob.deck.ny)
    assert _set_flux(gpu_lib, sim, flux) == -3
    assert b"several GPUs" in gpu_lib.nb200_last_error()
    sim.free()
    flux.free()


def test_deallocated_array_is_detached(gpu_lib):
    """6: after deallocate_data of the attached array, a freshly allocated array of the same
    size (often at the same address) stays zero through a timestep."""
    prob = build_problem("csp_small")
    sim = Simulation(prob, flux_tally=True)
    sim.inject()
    sim.step(1)
    gpu_lib.deallocate_data(sim.flux.ptr)
    sim.flux.ptr = None
    fresh = DeviceArray(sim.flux.n)
    sim.step(2)
    assert not np.any(fresh.download())
    fresh.free()
    sim.flux = None
    sim.free()


_TERMINATES = """
import sys
sys.path.insert(0, {root!r})
from neutral_b200.decks import build_problem
from neutral_b200.host import Simulation
sim = Simulation(build_problem("csp_small"), flux_tally=True)
sim.inject()
{change}
sim.step(1)
print("stepped")
"""


@pytest.mark.parametrize("change, message", [
    ("assert sim.lib.nb200_bank_set_flux_tally(sim.bank, sim.flux.ptr, sim.flux.n - 1) == 0",
     "the bank's flux tally has"),
    ("sim.lib.nb200_set_option(b'pipeline', 0)", "a flux tally needs pipeline=1"),
    ("sim.lib.nb200_set_option(b'tally_prereduce', 1)", "a flux tally needs pipeline=1"),
])
def test_enqueue_terminates(gpu_lib, change, message):
    """6: a mesh of another size than the attached array, or process-wide options turned to
    pipeline=0 / tally_prereduce=1 after attaching, end the process with the message."""
    res = subprocess.run([sys.executable, "-c", _TERMINATES.format(root=ROOT, change=change)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode != 0
    assert "stepped" not in res.stdout
    assert message in res.stderr, res.stderr
