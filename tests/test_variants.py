"""The oracle port, step by step, against the runs recorded in tests/golden/steps.json on problems
the reference decks do not cover (tests/variants.py): distinct capture/elastic tables (values
only, and grid + values), a coarse table, a rectangular non-uniform mesh, density boxes off the
tile grid. The recording is the port's own, which the UNMODIFIED reference library reproduced
bit for bit on every one of these problems; it pins the port there from now on."""
import numpy as np
import pytest

from recorded import field_hashes, reference_run, tally_matches_sample
from variants import VARIANTS


@pytest.mark.parametrize("name", list(VARIANTS))
def test_port_matches_reference_build_on_variant(port, name):
    prob = VARIANTS[name]()
    d = prob.deck
    want = reference_run(name)
    bank = port.inject(prob)
    assert field_hashes(bank) == want["hashes"][0], "inject"
    t_port = np.zeros(d.nx * d.ny)
    events = 0
    for tt in range(1, d.iterations + 1):
        pf, pc, _ = port.step(prob, bank, tt, t_port)
        assert [pf, pc] == want["counts"][tt - 1], f"step {tt}"
        assert field_hashes(bank) == want["hashes"][tt], f"step {tt}"
        assert abs(t_port.sum() - want["tally_sums"][tt - 1]) <= 1e-12 * abs(t_port.sum())
        events += pf + pc
    assert tally_matches_sample(t_port, name, 1e-12)
    # the variant must actually exercise both event kinds
    assert events > 10 * d.nparticles


def test_variants_break_the_reference_decks_symmetries():
    p = VARIANTS["absorb_scaled"]()
    assert np.array_equal(p.cs_scatter[0], p.cs_absorb[0])
    assert not np.array_equal(p.cs_scatter[1], p.cs_absorb[1])
    p = VARIANTS["absorb_own_grid"]()
    assert len(p.cs_scatter[0]) != len(p.cs_absorb[0])
    assert np.all(np.diff(p.cs_absorb[0]) > 0)
    p = VARIANTS["rect_stretched"]()
    assert p.deck.nx != p.deck.ny
    assert np.ptp(np.diff(p.edgex)) > 1e-3 and np.all(np.diff(p.edgex) > 0)
    assert np.all(np.diff(p.edgey) > 0)
    for name in ("rect_stretched", "multi_tile"):
        rho = VARIANTS[name]().density
        # at least one 16x16 tile holds more than one density value
        ny, nx = rho.shape
        mixed = any(np.unique(rho[y:y + 16, x:x + 16]).size > 1
                    for y in range(0, ny, 16) for x in range(0, nx, 16))
        assert mixed, name
