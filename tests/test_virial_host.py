"""CPU: the total-stress rows entry point (gprb_virial_rows) is declared, bound and exported, refuses bad arguments
before any CUDA call, and the Python gather refuses a descriptor without rdxdr."""
import ctypes

import pytest
import torch

from test_lib_symbols import _declared


def test_virial_rows_symbol_is_declared_bound_and_exported():
    from gpr_calculator_b200 import _lib
    assert "gprb_virial_rows" in _declared()
    assert "gprb_virial_rows" in _lib.SIGNATURES
    assert hasattr(_lib.load(), "gprb_virial_rows")


def test_virial_rows_rejects_bad_arguments():
    from gpr_calculator_b200 import _lib
    lib = _lib.load()
    buf = (ctypes.c_double * 8)()
    ints = (ctypes.c_int * 3)(0, 1, 2)
    p_i, p_d = ctypes.cast(ints, ctypes.c_void_p), ctypes.cast(buf, ctypes.c_void_p)
    null = ctypes.c_void_p(0)
    for n, d, sp, rd, out in ((2, 30, null, p_d, p_d), (2, 30, p_i, null, p_d), (2, 30, p_i, p_d, null),
                              (2, 0, p_i, p_d, p_d), (2, 65, p_i, p_d, p_d), (-1, 30, p_i, p_d, p_d)):
        assert lib.gprb_virial_rows(n, d, sp, rd, out, null) == _lib.ERR_ARG, (n, d)
        assert b"gprb_virial_rows" in lib.gprb_last_error()


def test_virial_rows_need_rdxdr():
    from gpr_calculator_b200.batch import virial_rows_from_batch
    r = {"x": torch.ones((2, 30), dtype=torch.float64), "rdxdr": None, "atom_ptr": torch.tensor([0, 2]),
         "seq_ptr": torch.tensor([0, 1, 2]), "numbers": torch.tensor([29, 29])}
    with pytest.raises(ValueError):
        virial_rows_from_batch(r)
