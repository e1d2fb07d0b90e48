"""The attention geometry helpers every kernel shares (dalle_pytorch_b200/csrc/attn_common.cuh: element predicate, 128-wide row /
column bit masks, tile-skip and tile-full tests, gathered-axial index maps and segment tiles) checked on the host: the header is
plain C++ apart from the CUDA keywords, so g++ compiles it against a stub `common.cuh` (tests/host/) and a driver walks a grid of
ragged geometries exhaustively (hundreds of thousands of tiles, every bit compared with the element predicate); the element
predicate itself is compared with the CPU oracle's `allowed_mask`, which tests/test_oracle_vs_golden.py pins to the reference's stored outputs.
The GPU tests can only sample geometries; a wrong bit here would be silently wrong attention for some (text_len, fmap, kernel)."""
import os
import shutil
import subprocess

import pytest
import torch

from dalle_oracle import allowed_mask

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def checker(tmp_path_factory):
    if shutil.which('g++') is None:
        pytest.skip('g++ not available')
    d = tmp_path_factory.mktemp('attn_geometry')
    shutil.copy(os.path.join(ROOT, 'dalle_pytorch_b200', 'csrc', 'attn_common.cuh'), d)
    shutil.copy(os.path.join(ROOT, 'tests', 'host', 'attn_geometry_check.cpp'), d)
    stub = open(os.path.join(ROOT, 'tests', 'host', 'common.cuh')).read()
    stub = stub.replace('"../../include/dalle_b200.h"', '"' + os.path.join(ROOT, 'include', 'dalle_b200.h') + '"')
    open(os.path.join(d, 'common.cuh'), 'w').write(stub)
    exe = os.path.join(d, 'attn_geometry_check')
    r = subprocess.run(['g++', '-O2', '-std=c++17', '-o', exe, os.path.join(d, 'attn_geometry_check.cpp')], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_bit_masks_tile_tests_and_gather_maps_exhaustively(checker):
    r = subprocess.run([checker], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith('OK '), r.stdout[-3000:]
    assert int(r.stdout.split()[1]) > 100000          # the grid really ran


@pytest.mark.parametrize('kind,code', [('full', 0), ('axial_row', 1), ('axial_col', 2), ('conv_like', 3)])
@pytest.mark.parametrize('T,fm,ks,dil', [(1, 1, 1, 1), (3, 4, 3, 1), (9, 5, 5, 1), (9, 6, 3, 2), (33, 8, 5, 2), (257, 32, 5, 1)])
def test_element_predicate_equals_the_pinned_oracle(checker, kind, code, T, fm, ks, dil):
    n = T + fm * fm - 1
    if n < 1:
        pytest.skip('empty sequence')
    r = subprocess.run([checker, 'dump', str(code), '1', str(T), str(fm), str(ks), str(dil), str(n)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0
    got = torch.tensor([[c == '1' for c in line] for line in r.stdout.split()], dtype=torch.bool)
    want = allowed_mask(kind, n, n, T, fm, True, ks, dil)
    assert got.shape == want.shape == (n, n)
    assert torch.equal(got, want), f'{int((got != want).sum())} entries differ'
