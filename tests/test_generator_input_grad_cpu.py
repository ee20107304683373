"""CPU checks of the generator's input-gradient entry points (srg_generator_forward_frozen, srg_generator_backward_ex):
the library exports them and rejects bad arguments before any CUDA call, so none of this needs a device."""
import ctypes
from ctypes import byref, c_void_p

import pytest

import srgan_b200 as S


@pytest.fixture(scope="module")
def L():
    return S.lib()


@pytest.fixture
def engine(L):
    h = c_void_p()
    assert L.srg_generator_create(byref(h), 2, 16, 24, 2, 2) == 0     # create() needs no device
    yield h
    L.srg_generator_destroy(h)


def _err(L) -> str:
    return L.srg_last_error().decode()


def test_library_exports_both_symbols():
    so = ctypes.CDLL(S._lib.SO_PATH)
    for name in ("srg_generator_forward_frozen", "srg_generator_backward_ex"):
        assert hasattr(so, name), name
        assert name in S._lib.EXPORTS, name


def test_backward_ex_rejects_an_unbound_engine(L, engine):
    dsr = ctypes.create_string_buffer(16)
    dlr = ctypes.create_string_buffer(16)
    assert L.srg_generator_backward_ex(engine, dsr, 1, dlr, None) != 0
    assert "workspace" in _err(L)
    assert L.srg_generator_backward_ex(engine, dsr, 1, None, None) != 0
    assert "workspace" in _err(L)


def test_backward_ex_rejects_a_null_gradient(L, engine):
    dlr = ctypes.create_string_buffer(16)
    assert L.srg_generator_backward_ex(engine, None, 1, dlr, None) != 0
    assert "null" in _err(L)


def test_backward_ex_rejects_a_request_for_nothing(L, engine):
    dsr = ctypes.create_string_buffer(16)
    assert L.srg_generator_backward_ex(engine, dsr, 0, None, None) != 0
    assert "nothing to compute" in _err(L)


def test_null_engine_is_rejected(L):
    buf = ctypes.create_string_buffer(16)
    assert L.srg_generator_backward_ex(None, buf, 1, buf, None) != 0
    assert "null engine" in _err(L)
    assert L.srg_generator_forward_frozen(None, buf, buf, None) != 0
    assert "null engine" in _err(L)


def test_forward_frozen_rejects_an_unbound_engine_and_null_images(L, engine):
    buf = ctypes.create_string_buffer(16)
    assert L.srg_generator_forward_frozen(engine, buf, buf, None) != 0
    assert "workspace" in _err(L)
    assert L.srg_generator_forward_frozen(engine, None, buf, None) != 0
    assert "null" in _err(L)
