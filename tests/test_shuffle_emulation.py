"""The CTA-parallel shuffle ALGORITHM (tests/emu_shuffle.py mirrors nhood_shuffle_cta_kernel step by step) against
numpy's Generator.shuffle, over sizes around powers of two, several thread counts and library segments."""

from __future__ import annotations

import random

import numpy as np
import pytest

from oracle import ref
from tests.emu_shuffle import emu_shuffle


def _state(seed):
    st = ref.spawn_states(seed, 1)[0]
    return st, (int(st[0]) << 64) | int(st[1]), (int(st[2]) << 64) | int(st[3])


@pytest.mark.parametrize("nt", [4, 32, 128])
def test_emulated_cta_shuffle_matches_numpy(nt):
    rnd = random.Random(nt)
    for n in [1, 2, 3, 4, 5, 8, 9, 16, 17, 33, 64, 65, 127, 128, 129, 255, 257, 1000, 1024, 1025, 4099]:
        seed = rnd.randrange(10**6)
        st, state, inc = _state(seed)
        gen = np.random.default_rng(np.random.SeedSequence(seed).spawn(1)[0])
        exp = np.arange(n, dtype=np.uint32)
        gen.shuffle(exp)
        got = emu_shuffle(list(range(n)), state, inc, [(0, n)], NT=nt, rng=rnd)
        np.testing.assert_array_equal(np.array(got, dtype=np.uint32), exp)


def test_emulated_cta_shuffle_segments():
    rnd = random.Random(7)
    for n in [10, 100, 513, 3000]:
        seed = rnd.randrange(10**6)
        st, state, inc = _state(seed)
        cuts = sorted(rnd.sample(range(1, n), 3))
        bounds = [0] + cuts + [n]
        segs = [(bounds[k], bounds[k + 1] - bounds[k]) for k in range(4)]
        exp = np.arange(n, dtype=np.uint32)
        s6 = st.copy()
        for b, m in segs:
            exp[b : b + m] = ref.shuffle_u32(s6, exp[b : b + m])
        got = emu_shuffle(list(range(n)), state, inc, segs, NT=16, rng=rnd)
        np.testing.assert_array_equal(np.array(got, dtype=np.uint32), exp)


def test_list_resolution_equals_serial_swaps():
    """The serial-pass-free conflict resolution of shuffle_algo 7 (tests/emu_shuffle.resolve_window_lists) against the
    plain in-order application of the same swaps, on windows far denser in conflicts than the device ever sees."""
    from tests.emu_shuffle import resolve_window_lists

    rnd = random.Random(11)
    for trial in range(3000):
        n = rnd.randrange(2, 80)
        i_cur = n - 1
        S = rnd.randrange(1, n)  # up to the whole array in one window
        mode = trial % 3
        sj = []
        for s in range(S):
            top = i_cur - s
            if mode == 0:
                sj.append(rnd.randrange(0, top + 1))
            elif mode == 1:  # mostly inside the window's own range
                sj.append(rnd.randrange(max(0, top - 6), top + 1))
            else:  # few distinct outside targets
                sj.append(min(top, rnd.randrange(0, 4)))
        base = rnd.randrange(0, 3)
        a0 = [rnd.randrange(1000) for _ in range(base + n)]
        exp = list(a0)
        for s in range(S):
            t, j = base + i_cur - s, base + sj[s]
            exp[t], exp[j] = exp[j], exp[t]
        got = list(a0)
        resolve_window_lists(got, base, i_cur, sj, rnd)
        assert got == exp, (trial, n, S, sj)


@pytest.mark.parametrize("nt", [4, 64])
def test_emulated_list_shuffle_matches_numpy(nt):
    rnd = random.Random(100 + nt)
    for n in [2, 3, 5, 17, 64, 129, 1000, 4099]:
        seed = rnd.randrange(10**6)
        st, state, inc = _state(seed)
        gen = np.random.default_rng(np.random.SeedSequence(seed).spawn(1)[0])
        exp = np.arange(n, dtype=np.uint32)
        gen.shuffle(exp)
        got = emu_shuffle(list(range(n)), state, inc, [(0, n)], NT=nt, rng=rnd, resolve="lists")
        np.testing.assert_array_equal(np.array(got, dtype=np.uint32), exp)


def _numpy_shuffle_from_targets(n, targets, base=0):
    a = np.arange(n, dtype=np.uint32)
    for i in range(n - 1, 0, -1):
        j = targets[(base, i)]
        a[i], a[j] = a[j], a[i]
    return a


@pytest.mark.parametrize("q", [2, 4])
def test_emulated_target_generation(q):
    """nhood_jgen_kernel's algorithm (tests/emu_shuffle.emu_targets): batch-sized windows and the one-pass acceptance when no
    candidate depends on its rank give numpy's swap targets — including small arrays, where most windows do need the fixed point."""
    from tests.emu_shuffle import emu_targets, serial_targets

    rnd = random.Random(40 + q)
    for n in [2, 3, 9, 33, 100, 257, 1000, 1025, 4099, 20011]:
        seed = rnd.randrange(10**6)
        st, state, inc = _state(seed)
        exp_t = serial_targets(state, inc, [(0, n)])
        gen = np.random.default_rng(np.random.SeedSequence(seed).spawn(1)[0])
        exp = np.arange(n, dtype=np.uint32)
        gen.shuffle(exp)
        np.testing.assert_array_equal(_numpy_shuffle_from_targets(n, exp_t), exp)  # the serial replay IS numpy's shuffle
        stats = {}
        got_t = emu_targets(state, inc, [(0, n)], Q=q, stats=stats)
        assert got_t == exp_t, (n, q)
        assert emu_targets(state, inc, [(0, n)], Q=q, shortcut=None) == exp_t
        if n >= 20011:
            assert stats["one_pass"] > 0  # the shortcut is actually taken on large arrays


def test_emulated_target_generation_segments_and_wrong_shortcut():
    from tests.emu_shuffle import emu_targets, serial_targets

    rnd = random.Random(9)
    st, state, inc = _state(77)
    segs = [(0, 700), (700, 1), (701, 2300), (3001, 40)]
    assert emu_targets(state, inc, segs, Q=4) == serial_targets(state, inc, segs)
    # the first version of the shortcut tested the current flags instead of the candidates: wrong on small arrays
    wrong = 0
    for trial in range(40):
        st, state, inc = _state(rnd.randrange(10**6))
        n = rnd.choice([300, 1000, 1500])
        wrong += emu_targets(state, inc, [(0, n)], Q=4, shortcut="flags") != serial_targets(state, inc, [(0, n)])
    assert wrong > 0


def _fisher_yates(arr, J):
    a = list(arr)
    for i in range(len(a) - 1, 0, -1):
        j = J[i]
        a[i], a[j] = a[j], a[i]
    return a


def test_region_replay_equals_fisher_yates():
    """The region replay (tests/emu_shuffle.region_replay = the specification of nhood_apply_region_kernel, last present in
    commit eef2f18): applying every step in the pass of the region its TARGET falls into -- tops above the region through
    compacted windows, tops inside through consecutive windows, targets below deferred with T(step) left at the top -- equals
    the plain Fisher-Yates sweep, for any region size, window size and target distribution (uniform like the real stream, and
    adversarial: many duplicates, many own-range targets, all targets in one region)."""
    from tests.emu_shuffle import region_replay

    rnd = random.Random(5)
    stats = {}
    for trial in range(1500):
        m = rnd.choice([2, 3, 5, 17, 40, 97, 200, 333])
        mode = trial % 4
        J = [0] * m
        for i in range(1, m):
            if mode == 0:
                J[i] = rnd.randrange(i + 1)
            elif mode == 1:  # few distinct targets: long duplicate lists
                J[i] = min(i, rnd.choice([0, 1, 2, m // 3, m // 2]))
            elif mode == 2:  # targets close to the top: own-range chains
                J[i] = max(0, i - rnd.randrange(0, 4))
            else:  # everything aims at the lowest positions: every region defers almost all of its steps
                J[i] = rnd.randrange(min(i + 1, 6))
        arr = [rnd.randrange(1000) for _ in range(m)]
        cap = rnd.choice([16, 32, 48, 64, 128, 1024])
        nt = rnd.choice([4, 8, 16])
        got = region_replay(arr, J, cap, NT=nt, WL=rnd.choice([2, 4]), CAPW=rnd.choice([8, 12]), KMAX=rnd.choice([2, 16]), rng=rnd, stats=stats)
        assert got == _fisher_yates(arr, J), (trial, m, cap, nt, mode)
    assert stats.get("xwin", 0) > 1000 and stats.get("overflow", 0) > 0  # compacted windows and the halving path were exercised
