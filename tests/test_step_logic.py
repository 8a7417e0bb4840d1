"""The play step's board and policy helpers on the host (tests/host_shim/step_logic.cpp): the spawn's 2/4 decision as one
compare, the transpose and row mirror in 32-bit halves, and the random policy's action from the legal-mask table."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("step_logic") / "libstep_logic.so"
    src = ROOT / "tests" / "host_shim" / "step_logic.cpp"
    res = subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-w", "-o", str(out), str(src)],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]
    return C.CDLL(str(out))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _unpack(x):
    return ((x[:, None] >> (np.arange(16, dtype=np.uint64) * np.uint64(4))) & np.uint64(15)).astype(np.uint64)


def _pack(cells):
    return (cells.astype(np.uint64) << (np.arange(16, dtype=np.uint64) * np.uint64(4))).sum(1).astype(np.uint64)


def test_spawn_four_compare_over_all_draws():
    """m = 2^23 - (bits >> 9) > 7549747 (1 - u > 0.9f) <=> bits < 429496832, for all 2^23 values of bits >> 9."""
    h = np.arange(1 << 23, dtype=np.uint64)
    old = (np.uint64(0x800000) - h) > np.uint64(7549747)
    for low in (0, 511):
        assert np.array_equal(old, ((h << np.uint64(9)) | np.uint64(low)) < np.uint64(429496832))


def test_spawn_select_value_over_all_draws(lib):
    """spawn_select's exponent against the original form of the decision, for all 2^23 values of bits >> 9."""
    h = np.arange(1 << 23, dtype=np.int64)
    want = np.where((0x800000 - h) > 7549747, 2, 1).astype(np.uint8)
    for low in (0, 511):
        got = np.zeros(1 << 23, np.uint8)
        lib.step_spawn_val_all(C.c_uint32(low), _p(got))
        np.testing.assert_array_equal(got, want)


def test_transpose_and_mirror(lib):
    rng = np.random.default_rng(5)
    boards = np.concatenate([rng.integers(0, 1 << 63, 20000, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, 20000, dtype=np.uint64),
                             np.array([0, 0xFFFFFFFFFFFFFFFF, 0x0123456789ABCDEF, 0xFEDCBA9876543210], np.uint64)])
    n = boards.shape[0]
    t, m = np.zeros(n, np.uint64), np.zeros(n, np.uint64)
    lib.step_transpose_mirror(_p(boards), C.c_int64(n), _p(t), _p(m))
    cells = _unpack(boards).reshape(n, 4, 4)
    np.testing.assert_array_equal(t, _pack(cells.transpose(0, 2, 1).reshape(n, 16)))
    np.testing.assert_array_equal(m, _pack(cells[:, :, ::-1].reshape(n, 16)))


def test_action_table_matches_argmax(lib):
    """act_random_table (bits & mm + c, max, ~max & 7) picks what argmax_bits_legal picks: the first allowed action with
    the largest bits >> 9, all four when no action is legal -- for every legal mask, with ties in bits >> 9."""
    rng = np.random.default_rng(11)
    k = 20000
    rand = rng.integers(0, 1 << 32, (k, 4), dtype=np.uint64).astype(np.uint32)
    # ties: the same bits >> 9 on a random subset of the actions, different low bits
    tie = rng.integers(0, 1 << 32, (k, 1), dtype=np.uint64).astype(np.uint32) & np.uint32(0xFFFFFE00)
    tied = np.where(rng.integers(0, 2, (k, 4)).astype(bool), tie | rng.integers(0, 512, (k, 4)).astype(np.uint32), rand)
    edge = np.array([[0, 0, 0, 0], [0xFFFFFFFF] * 4, [511, 0, 0, 0], [0, 0, 0, 0xFFFFFFFF], [0x200, 0x1FF, 0x3FF, 0]], np.uint32)
    bits = np.concatenate([rand, tied, edge])
    bits = np.repeat(bits, 16, axis=0)
    lm = np.tile(np.arange(16, dtype=np.uint32), bits.shape[0] // 16)
    n = bits.shape[0]
    got, ref = np.zeros(n, np.int32), np.zeros(n, np.int32)
    lib.step_act(_p(np.ascontiguousarray(bits)), _p(lm), C.c_int64(n), _p(got), _p(ref))
    np.testing.assert_array_equal(got, ref)
    allowed = np.where(lm == 0, 15, lm)
    assert np.all((allowed >> ref.astype(np.uint32)) & 1)  # never an illegal action while a legal one exists
