"""The batched flux's entry points without a GPU: each checks its handle before it needs a
device, and the Python binding declares them."""
import ctypes as C

from neutral_b200.bank import ParticleSoA
from neutral_b200.host import EXPORTED_SYMBOLS


def test_batched_flux_entry_points_refuse_a_non_bank_without_a_device(lib):
    junk = (C.c_double * 16)()
    handle = C.cast(C.addressof(junk), C.POINTER(ParticleSoA))
    total = C.c_double(0.0)
    calls = {
        "nb200_bank_set_batched_flux_tally": lambda h: lib.nb200_bank_set_batched_flux_tally(
            h, C.addressof(junk), 16),
        "nb200_bank_flux_batches": lambda h: lib.nb200_bank_flux_batches(h, C.addressof(junk), 16),
        "nb200_bank_flux_relerr": lambda h: lib.nb200_bank_flux_relerr(h, C.addressof(junk),
                                                                        C.byref(total)),
    }
    for name, call in calls.items():
        assert name in EXPORTED_SYMBOLS
        for h in (handle, None):
            assert call(h) == -3, name
            assert b"not a bank handle" in lib.nb200_last_error(), name
    assert lib.nb200_bank_set_batched_flux_tally(None, None, 0) == -3
    assert total.value == 0.0
