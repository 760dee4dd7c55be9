"""The tile-level symbolic Cholesky fill of the large-window BA solve (ov2slam_b200/csrc/ba_fill.cuh), compiled for the host
on its own: the tiles the keyframe block pattern covers, closed under the right-looking update, against a dense numpy
symbolic Cholesky.  The factorisation (csrc/ba_large.cu) zeroes, accumulates, factors and updates only these tiles, so the
set must also cover every tile in which the scalar-level factor can be non-zero."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
TILE = 32

_SRC = r'''
#include "%s/ov2slam_b200/csrc/ba_fill.cuh"
extern "C" void tile_fill(int nt, int npair, const int* pairs, uint8_t* T) {
    for (int p = 0; p < npair; ++p) bafill::mark_block(nt, T, pairs[2 * p], pairs[2 * p + 1]);
    bafill::symbolic_fill(nt, T);
}
extern "C" int tile_size() { return bafill::TILE; }
'''


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("fill")
    src, so = d / "fill.cpp", d / "libfill.so"
    src.write_text(_SRC % ROOT)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", str(so), str(src)])
    L = C.CDLL(str(so))
    L.tile_fill.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    assert L.tile_size() == TILE
    return L


def _fill_c(lib, ncv, blocks):
    nt = max(1, -(-6 * ncv // TILE))
    T = np.zeros((nt, nt), np.uint8)
    pairs = np.ascontiguousarray(np.array(sorted(blocks), np.int32).reshape(-1, 2))
    lib.tile_fill(nt, len(pairs), pairs.ctypes.data, T.ctypes.data)
    return np.triu(T).astype(bool)


def _symbolic_cholesky(M):
    """Dense symbolic right-looking Cholesky of a symmetric boolean pattern (upper triangle returned)."""
    M = np.triu(M | M.T).copy()
    np.fill_diagonal(M, True)
    for k in range(len(M)):
        j = k + 1 + np.nonzero(M[k, k + 1:])[0]
        if len(j) > 1:
            M[np.ix_(j, j)] = True
    return np.triu(M)


def _tiles_of(scalar, nt):
    n = scalar.shape[0]
    pad = np.zeros((nt * TILE, nt * TILE), bool)
    pad[:n, :n] = scalar
    return np.triu(pad.reshape(nt, TILE, nt, TILE).any(axis=(1, 3)))


def _reference(ncv, blocks, scalar=True):
    n = 6 * ncv
    nt = max(1, -(-n // TILE))
    S = np.zeros((n, n), bool)
    for lo, hi in blocks:
        S[6 * lo:6 * lo + 6, 6 * hi:6 * hi + 6] = True
    S = np.triu(S | S.T)
    tiles = _tiles_of(S, nt)                           # tiles the accumulation touches
    return _symbolic_cholesky(tiles), (_tiles_of(_symbolic_cholesky(S), nt) if scalar else None)


def _random_blocks(rng, ncv, density):
    B = np.triu(rng.random((ncv, ncv)) < density)
    np.fill_diagonal(B, True)
    return [(int(i), int(j)) for i, j in zip(*np.nonzero(B))]


def _band_loop_blocks(ncv, band, loop):
    """A trajectory: every keyframe coupled to the next `band`, and the last `loop` keyframes to the first `loop`."""
    out = set()
    for i in range(ncv):
        for j in range(i, min(ncv, i + band + 1)):
            out.add((i, j))
    for i in range(loop):
        for j in range(ncv - loop, ncv):
            out.add((min(i, j), max(i, j)))
    return sorted(out)


@pytest.mark.parametrize("seed,ncv,density", [(0, 5, 0.3), (1, 70, 0.02), (2, 160, 0.01), (3, 300, 0.004), (4, 96, 0.2)])
def test_tile_fill_equals_dense_symbolic_cholesky_random(lib, seed, ncv, density):
    rng = np.random.default_rng(seed)
    blocks = _random_blocks(rng, ncv, density)
    got = _fill_c(lib, ncv, blocks)
    tiles_fill, scalar_fill = _reference(ncv, blocks)
    assert np.array_equal(got, tiles_fill)
    assert not (scalar_fill & ~got).any()              # every tile the factor can fill is in the set


@pytest.mark.parametrize("ncv,band,loop", [(65, 3, 4), (160, 5, 6), (300, 6, 8), (1024, 6, 10), (120, 2, 0)])
def test_tile_fill_equals_dense_symbolic_cholesky_band_plus_loop(lib, ncv, band, loop):
    blocks = _band_loop_blocks(ncv, band, loop)
    got = _fill_c(lib, ncv, blocks)
    tiles_fill, scalar_fill = _reference(ncv, blocks, scalar=ncv <= 300)
    assert np.array_equal(got, tiles_fill)
    assert scalar_fill is None or not (scalar_fill & ~got).any()
    nt = got.shape[0]
    if loop == 0:
        assert got.sum() < 3 * nt                      # a pure band stays a band of tiles
    assert got.sum() < nt * (nt + 1) // 2 or nt <= 2 * (band + loop)
