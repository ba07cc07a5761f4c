"""Host logic around the hot path: deck reader, mesh, density painting, source box and the
regenerated cross-section table - checked against the C arch-lite shim the reference driver
is built on and against facts of the reference's own decks/tables."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

from neutral_b200 import decks
from neutral_b200.decks import (CS_TABLE_MD5, build_problem, cross_section_table,
                                cross_section_text, load_deck)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    """archlite compiled as a host shared library."""
    out = tmp_path_factory.mktemp("shim") / "libarchlite.so"
    src = [os.path.join(ROOT, "archlite", f) for f in ("archlite.c", "alloc_host.c")]
    subprocess.run(["gcc", "-O1", "-std=gnu99", "-ffp-contract=off", "-fPIC", "-shared",
                    "-DENABLE_PROFILING", "-I", os.path.join(ROOT, "archlite")] + src +
                   ["-o", str(out), "-lm"], check=True)
    return C.CDLL(str(out))


class Mesh(C.Structure):  # archlite/mesh.h
    _fields_ = [(n, C.c_int) for n in
                ("global_nx", "global_ny", "global_nz", "local_nx", "local_ny", "local_nz",
                 "pad", "x_off", "y_off", "z_off", "niters", "rank", "nranks", "ndims")] + \
               [("neighbours", C.c_int * 6)] + \
               [(n, C.c_double) for n in ("width", "height", "depth", "dt", "dt_h", "sim_end",
                                          "max_dt")] + \
               [(n, C.POINTER(C.c_double)) for n in ("edgex", "edgey", "edgedx", "edgedy")]


class SharedData(C.Structure):  # archlite/shared_data.h
    _fields_ = [("density", C.POINTER(C.c_double)), ("energy", C.POINTER(C.c_double))]


def test_cross_section_table_is_the_reference_table():
    txt = cross_section_text()
    assert hashlib.md5(txt).hexdigest() == CS_TABLE_MD5
    keys, values = cross_section_table()
    assert len(keys) == 29999 and keys[0] == 1.000000012347e-02 and keys[-1] == 1.0000000001e8
    assert values[0] == 1001.0 and np.all(np.diff(values) < 0)


# source box and density boxes (density, x, y, width, height) of the reference's own decks
REFERENCE_DECK_BOXES = {
    "scatter": ((0.2, 0.2, 0.6, 0.6), [(1.0e4, 0.0, 0.0, 1.0, 1.0)]),
    "stream": ((0.45, 0.45, 0.1, 0.1), [(1.0e-30, 0.0, 0.0, 1.0, 1.0)]),
    "csp": ((0.1, 0.1, 0.2, 0.2), [(1.0e-30, 0.0, 0.0, 1.0, 1.0), (1.0e4, 0.4, 0.4, 0.2, 0.2)]),
    "split": ((0.4, 0.4, 0.2, 0.2), [(1.0e-30, 0.0, 0.0, 1.0, 0.5), (1.0e3, 0.0, 0.5, 1.0, 0.5)]),
}


@pytest.mark.parametrize("name,nparticles,energy,iters", [
    ("scatter", 10_000_000, 1.0e3, 2), ("stream", 1_000_000, 1.0e6, 1),
    ("csp", 1_000_000, 1.0e4, 10), ("split", 1_000_000, 2.5e4, 1)])
def test_baseline_decks(name, nparticles, energy, iters):
    d = load_deck(name)
    assert (d.nx, d.ny, d.dt) == (4000, 4000, 1.0e-7)
    assert (d.nparticles, d.initial_energy, d.iterations) == (nparticles, energy, iters)
    assert (d.source, d.problems) == REFERENCE_DECK_BOXES[name]


@pytest.mark.parametrize("name", ["csp_small", "split_small", "mixed_small", "csp"])
def test_python_setup_equals_c_shim(shim, name):
    prob = build_problem(name)
    d = prob.deck
    m = Mesh()
    m.global_nx, m.global_ny, m.local_nx, m.local_ny = d.nx, d.ny, d.nx, d.ny
    m.pad = m.x_off = m.y_off = 0
    m.width, m.height = d.width, d.height
    shim.initialise_mesh_2d(C.byref(m))
    ex = np.ctypeslib.as_array(m.edgex, shape=(d.nx + 1,))
    ey = np.ctypeslib.as_array(m.edgey, shape=(d.ny + 1,))
    assert np.array_equal(ex, prob.edgex) and np.array_equal(ey, prob.edgey)
    sd = SharedData()
    shim.initialise_shared_data_2d.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double,
                                               C.c_double, C.c_char_p, C.POINTER(C.c_double),
                                               C.POINTER(C.c_double), C.POINTER(SharedData)]
    shim.initialise_shared_data_2d(d.nx, d.ny, 0, d.width, d.height, d.path.encode(), m.edgex,
                                   m.edgey, C.byref(sd))
    rho = np.ctypeslib.as_array(sd.density, shape=(d.ny, d.nx))
    assert np.array_equal(rho, prob.density)
    shim.get_int_parameter.argtypes = [C.c_char_p, C.c_char_p]
    shim.get_double_parameter.argtypes = [C.c_char_p, C.c_char_p]
    shim.get_double_parameter.restype = C.c_double
    assert shim.get_int_parameter(b"nparticles", d.path.encode()) == d.nparticles
    assert shim.get_double_parameter(b"initial_energy", d.path.encode()) == d.initial_energy


def test_source_box_csp():
    prob = build_problem("csp")
    s = prob.source
    assert s.nlocal_particles == 1_000_000
    assert s.left == 0.1 and s.bottom == 0.1
    assert abs(s.width - 0.2) < 1e-15 and abs(s.height - 0.2) < 1e-15
    assert np.count_nonzero(prob.density == 1.0e4) == 641601  # 801 x 801 cells


def test_neutral_tests_entries():
    tests = os.path.join(ROOT, "problems", "neutral.tests")
    kv = decks.get_key_value_parameter("problems/csp.params", tests)
    assert kv == [("result", 1.121870290714e+07)]
