"""The structured prune -> line quantize step's entry points reject bad arguments before any CUDA call (no GPU in
this tier: the pointers are host buffers that are never dereferenced)."""
import ctypes

import pytest

QSB_E_BADARG, QSB_E_UNSUPPORTED = -1, -4


@pytest.fixture(scope="module")
def lib():
    from qsparse_b200 import _native
    return _native.load_library()


C = 8


@pytest.fixture()
def bufs():
    f = lambda n: (ctypes.c_float * n)()
    return dict(x=f(64 * C), ws=(ctypes.c_uint8 * 4096)(), arrival=(ctypes.c_uint32 * 64)(), mag=f(C),
                mask=(ctypes.c_uint8 * C)(), lines=f(2 * C), counter=(ctypes.c_int64 * 1)(), group=(ctypes.c_uint8 * 64)())


def one_launch(lib, b, channels=C, n_lines=C, t_line=1, k=2, refresh=1, counter=False, group=False, lines=True,
               mask=True, x=True, mode=1, count=64.0, dtype=0):
    return lib.qsb_reduce_prune_line_step_dt(
        b["x"] if x else None, dtype, 64, channels, 1, b["ws"], 4096, b["arrival"], b["mag"],
        b["mask"] if mask else None, b["lines"] if lines else None, n_lines, b["group"] if group else None, count, 1,
        mode, refresh, k, t_line, None, None, None, b["counter"] if counter else None, None)


def partials(lib, b, channels=C, n_lines=C, t_line=1, k=2, refresh=1, counter=False, group=False, lines=True,
             mask=True):
    return lib.qsb_prune_line_step_params(
        b["mag"], b["mask"] if mask else None, b["lines"] if lines else None, n_lines, b["ws"], 4096, 64, channels,
        1, b["group"] if group else None, 64.0, 1, 1, refresh, k, t_line, None, None, None,
        b["counter"] if counter else None, None)


@pytest.mark.parametrize("call", [one_launch, partials], ids=["one-launch", "partials"])
def test_line_step_argument_errors(lib, bufs, call):
    assert call(lib, bufs, lines=False) == QSB_E_BADARG                  # NULL lines
    assert call(lib, bufs, mask=False) == QSB_E_BADARG                   # NULL mask
    assert call(lib, bufs, n_lines=2) == QSB_E_BADARG                    # n_lines neither 1 nor C
    assert call(lib, bufs, n_lines=0) == QSB_E_BADARG
    assert call(lib, bufs, t_line=0) == QSB_E_BADARG                     # t_line < 1 without a counter
    assert call(lib, bufs, k=C) == QSB_E_BADARG                          # k outside [0, C) on a refresh
    assert call(lib, bufs, k=-1) == QSB_E_BADARG
    assert call(lib, bufs, group=True) == QSB_E_BADARG                   # the line form takes no peer group
    assert call(lib, bufs, channels=0) == QSB_E_BADARG


def test_one_launch_argument_errors(lib, bufs):
    assert one_launch(lib, bufs, x=False) == QSB_E_BADARG
    assert one_launch(lib, bufs, dtype=7) == QSB_E_BADARG
    assert one_launch(lib, bufs, mode=3) == QSB_E_BADARG
    assert one_launch(lib, bufs, count=0.0) == QSB_E_BADARG
    assert one_launch(lib, bufs, channels=1025, n_lines=1) == QSB_E_UNSUPPORTED   # above the one-launch route


def test_partials_channel_limit(lib, bufs):
    assert partials(lib, bufs, channels=2049, n_lines=1) == QSB_E_UNSUPPORTED


def test_line_partials_argument_errors(lib, bufs):
    assert lib.qsb_reduce_line_partials_dt(None, 0, 64, C, 1, bufs["ws"], 4096, None) == QSB_E_BADARG
    assert lib.qsb_reduce_line_partials_dt(bufs["x"], 7, 64, C, 1, bufs["ws"], 4096, None) == QSB_E_BADARG
    assert lib.qsb_reduce_line_partials_dt(bufs["x"], 0, 0, C, 1, bufs["ws"], 4096, None) == QSB_E_BADARG
