"""CPU: the plumbing of uint16 count storage (ORI_F_X_U16) -- flag, row pitch, problem description, ingest selection."""
import os
import re

import numpy as np
import torch

from oriana_b200 import _lib
from oriana_b200.problem import build_problem, row_pitch
from oriana_b200.singlecell.cmatrix import CountMatrix

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_flag_matches_header():
    header = open(os.path.join(ROOT, 'include', 'oriana_b200.h')).read()
    m = re.search(r'#define ORI_F_X_U16 (\d+)u', header)
    assert m and int(m.group(1)) == _lib.ORI_F_X_U16 == 512
    flags = [int(v) for v in re.findall(r'#define ORI_F_\w+ (\d+)u', header)]
    assert len(set(flags)) == len(flags) and all(f & (f - 1) == 0 for f in flags)     # distinct single bits


def test_row_pitch_for_two_byte_counts():
    assert row_pitch(1, 2) == 8 and row_pitch(8, 2) == 8 and row_pitch(9, 2) == 16 and row_pitch(20001, 2) == 20008
    assert [row_pitch(p) for p in (1, 4, 5, 20001)] == [4, 4, 8, 20004]       # float32 unchanged
    for p in range(1, 70):
        assert row_pitch(p, 2) * 2 % 16 == 0 and 0 <= row_pitch(p, 2) - p < 8


def test_build_problem_with_uint16_counts():
    X = torch.zeros((3, row_pitch(13, 2)), dtype=torch.int16).view(torch.uint16)
    P = build_problem(n_rows=3, n_total=3, ldx=row_pitch(13, 2), p=13, K=2, KP=8, flags=_lib.ORI_F_X_U16, X=X)
    assert P.X == X.data_ptr() and P.ldx == 16 and P.flags & _lib.ORI_F_X_U16


def test_uint16_storage_only_where_float32_does_not_fit():
    from oriana_b200.problem import counts_storage
    n, p, KP = 2_000_000, 30_000, 64                                   # config 5: 240 GB of counts as float32
    gb = 10 ** 9
    assert counts_storage(True, n, p, KP, 178 * gb) == torch.uint16
    assert counts_storage(True, n, p, KP, 300 * gb) == torch.float32
    assert counts_storage(False, n, p, KP, 178 * gb) == torch.float32  # only uint16 inputs are ever kept as uint16
    assert counts_storage(True, 1_000_000, 20_000, 32, 178 * gb) == torch.float32   # config 4: 80 GB fits as float32


def test_uint16_selection_follows_the_dtype():
    X = np.arange(12).reshape(3, 4)
    assert CountMatrix(X.astype(np.uint16)).is_uint16()
    assert CountMatrix(torch.from_numpy(X.astype(np.uint16))).is_uint16()
    for dt in (np.float32, np.float64, np.int64, np.uint8, np.int16):
        assert not CountMatrix(X.astype(dt)).is_uint16(), dt
    blk = CountMatrix(X.astype(np.uint16)).row_block(1, 2)                   # sharding keeps the dtype
    assert blk.is_uint16() and blk.as_array().dtype == np.uint16
    assert CountMatrix(X.astype(np.uint16)).as_array().dtype == np.uint16
