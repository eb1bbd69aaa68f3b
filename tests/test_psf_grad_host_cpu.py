"""Host-side checks of the backward entry points of local_psf_render / render_psf_map (no GPU needed): argument
validation runs before any device call, and the PSF-map workspace size follows the forward's tiling."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    import aadff_b200
    return aadff_b200.native.lib


def bounds(grid, n):
    return (ctypes.c_int * (grid + 1))(*[int(i / grid * n) for i in range(grid + 1)])


def test_local_psf_render_backward_rejects_bad_arguments(lib):
    bwd = lib.aadff_local_psf_render_backward_f32
    assert bwd(None, 8, 8, 8, 8, 1, 3, 8, 8, 11, None) == -1
    assert b"null" in lib.aadff_last_error()
    assert bwd(8, 8, None, 8, 8, 1, 3, 8, 8, 11, None) == -1
    assert bwd(8, 8, 8, None, None, 1, 3, 8, 8, 11, None) == -1           # neither gradient requested
    assert bwd(8, 8, 8, 8, None, 1, 3, 8, 8, 10, None) == -1              # even kernel size
    assert b"kernel size" in lib.aadff_last_error()
    assert bwd(8, 8, 8, None, 8, 1, 0, 8, 8, 11, None) == -1              # no channel
    assert bwd(8, 8, 8, 8, 8, 0, 3, 8, 8, 11, None) == 0                  # empty batch: nothing to do


def test_render_psf_map_backward_rejects_bad_arguments(lib):
    bwd = lib.aadff_render_psf_map_backward_f32
    hb, wb = bounds(2, 16), bounds(2, 16)
    assert bwd(None, 8, 8, 8, 8, 8, 1 << 20, 1, 3, 16, 16, 3, 2, hb, wb, None) == -1
    assert bwd(8, 8, 8, None, None, None, 0, 1, 3, 16, 16, 3, 2, hb, wb, None) == -1
    assert bwd(8, 8, 8, None, 8, None, 1 << 20, 1, 3, 16, 16, 3, 2, hb, wb, None) == -1      # PSF gradient, no work
    assert bwd(8, 8, 8, 8, None, None, 0, 1, 3, 16, 16, 33, 2, hb, wb, None) == -1           # ks > 31
    assert bwd(8, 8, 8, 8, None, None, 0, 1, 3, 16, 16, 3, 33, bounds(33, 16), bounds(33, 16), None) == -1
    assert bwd(8, 8, 8, 8, None, None, 0, 1, 3, 4, 16, 11, 1, bounds(1, 4), bounds(1, 16), None) == -1  # p >= H
    assert b"reflect" in lib.aadff_last_error()
    bad = (ctypes.c_int * 3)(0, 9, 8)
    assert bwd(8, 8, 8, 8, None, None, 0, 1, 3, 16, 16, 3, 2, bad, wb, None) == -1
    need = lib.aadff_render_psf_map_backward_work_bytes(1, 3, 16, 16, 3, 2, hb, wb)
    assert bwd(8, 8, 8, None, 8, 8, need - 4, 1, 3, 16, 16, 3, 2, hb, wb, None) == -1
    assert b"workspace" in lib.aadff_last_error()


def test_render_psf_map_backward_work_bytes(lib):
    ws = lib.aadff_render_psf_map_backward_work_bytes
    # one ks^2 partial per (channel, cell, image, 32x64 tile of the largest cell)
    assert ws(2, 3, 100, 130, 11, 1, bounds(1, 100), bounds(1, 130)) == 3 * 1 * 2 * (4 * 3) * 121 * 4
    assert ws(1, 3, 70, 101, 3, 3, bounds(3, 70), bounds(3, 101)) == 3 * 9 * 1 * (1 * 1) * 9 * 4
    assert ws(1, 3, 16, 16, 3, 1, None, None) == -1
    assert ws(1, 3, 16, 16, 4, 1, bounds(1, 16), bounds(1, 16)) == -1
