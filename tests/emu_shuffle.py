"""Python emulation of the CTA-parallel exact numpy-shuffle replay implemented in squidpy_b200/csrc/nhood.cu.

It mirrors the device algorithm phase by phase (RNG batch by jump-ahead, windowed acceptance fixed point,
hash-based conflict detection, parallel swaps + ordered serial pass) so the *algorithm* can be validated on
the CPU against numpy's ``Generator.shuffle`` (tests/test_shuffle_emulation.py).  Not used by the product.

Also here: ``resolve_window_lists`` (the serial-pass-free conflict resolution of shuffle_algo 7) and ``emu_targets``
(nhood_jgen_kernel: batch-sized windows, one-pass acceptance), each the executable specification of its kernel.
"""
from __future__ import annotations

import math
import random

A = 0x2360ED051FC65DA44385DF649FCCF645
M128 = (1 << 128) - 1
M64 = (1 << 64) - 1


def _jump_consts(d):
    M, C = A, 1
    Mt, Ct = 1, 0
    while d:
        if d & 1:
            Mt, Ct = (M * Mt) & M128, (M * Ct + C) & M128
        M, C = (M * M) & M128, (M * C + C) & M128
        d >>= 1
    return Mt, Ct


def _out(s):
    hi, lo = s >> 64, s & M64
    x = hi ^ lo
    rot = hi >> 58
    return ((x >> rot) | (x << ((-rot) & 63))) & M64


def window_size(i_cur, raw_left, raw_total):
    """K: number of raw values examined per acceptance window (mirrors sqb_window_size in nhood.cu)."""
    k = min(i_cur // 4, int(4.0 * math.sqrt(float(i_cur))))
    k = max(1, min(k, raw_total))
    return min(k, raw_left)


def resolve_window_lists(a, base, i_cur, sj, rng):
    """Conflict resolution WITHOUT a serial pass (shuffle_algo 7, nhood_apply_list_kernel): applies the window's steps
    s = 0..S-1 (swap positions i_cur-s and sj[s]) to `a` in place.  Every step pushes itself on the list of the position
    it targets (arbitrary push order = thread interleaving); afterwards each step derives what it has to write from the
    lists alone, reading only ORIGINAL values:
      T(s) = value of the top position i_cur-s just before step s = T(latest earlier step targeting it) or the original;
      step s writes  a[top_s] = value of position sj[s] just before step s = T(latest earlier step targeting sj[s]) or original;
      the last step targeting an outside position p writes a[p] = T(that step)."""
    S = len(sj)
    own_lo = i_cur - S
    otop = [a[base + i_cur - s] for s in range(S)]          # staged original tops
    own_list = [[] for _ in range(S)]                        # steps targeting top position of step u (excluding u itself)
    tab = {}                                                 # outside target -> list of steps
    order = list(range(S))
    rng.shuffle(order)
    for s in order:
        j = sj[s]
        if j > own_lo:
            u = i_cur - j
            if u != s:
                own_list[u].append(s)
        else:
            tab.setdefault(j, []).append(s)
    orig_j = {j: a[base + j] for j in tab}

    def T(x):
        while own_list[x]:
            x = max(own_list[x])
        return otop[x]

    def latest_before(lst, s):
        c = [e for e in lst if e < s]
        return max(c) if c else None

    writes = []
    for s in order:
        j = sj[s]
        top = base + i_cur - s
        if j > own_lo:
            u = i_cur - j
            if u == s:
                writes.append((top, T(s)))
            else:
                p = latest_before(own_list[u], s)
                writes.append((top, T(p) if p is not None else otop[u]))
        else:
            lst = tab[j]
            p = latest_before(lst, s)
            writes.append((top, T(p) if p is not None else orig_j[j]))
            if s == max(lst):
                writes.append((base + j, T(s)))
    for pos, v in writes:
        a[pos] = v


def emu_shuffle(arr, state, inc, segs, NT=8, rng=None, stats=None, resolve="serial"):
    """arr: list (group-contiguous); segs: list of (start, length).  Returns shuffled list."""
    a = list(arr)
    RAW = 2 * NT
    rng = rng or random.Random(0)
    Mn, Cn = _jump_consts(NT)
    # thread t starts at state_{t+1}
    st = []
    for t in range(NT):
        Mt, Ct = _jump_consts(t + 1)
        st.append((Mt * state + Ct * inc) & M128)
    raw = [0] * RAW
    pos = RAW  # force generation

    def gen():
        nonlocal pos
        for t in range(NT):
            o = _out(st[t])
            raw[2 * t] = o & 0xFFFFFFFF
            raw[2 * t + 1] = o >> 32
            st[t] = (Mn * st[t] + Cn * inc) & M128
        pos = 0

    for (base, m) in segs:
        i_cur = m - 1
        while i_cur >= 1:
            if pos == RAW:
                gen()
            mask = (1 << i_cur.bit_length()) - 1
            i_lo = (mask >> 1) + 1
            n_ph = i_cur - i_lo + 1
            K = window_size(i_cur, RAW - pos, RAW)
            win = list(range(pos, pos + K))
            u = {r: raw[r] & mask for r in win}
            # fixed point on acceptance flags
            c = {r: 0 for r in win}
            F = {r: u[r] <= i_cur - c[r] for r in win}
            iters = 0
            while True:
                iters += 1
                run = 0
                for r in win:  # exclusive prefix of F
                    c[r] = run
                    run += 1 if F[r] else 0
                F2 = {r: u[r] <= i_cur - c[r] for r in win}
                if F2 == F:
                    break
                F = F2
            total = sum(F.values())
            if stats is not None:
                stats["iters"] = stats.get("iters", 0) + iters
                stats["windows"] = stats.get("windows", 0) + 1
            if total >= n_ph:
                S = n_ph
                rstar = next(r for r in win if F[r] and c[r] == n_ph - 1)
                newpos = rstar + 1
            else:
                S = total
                newpos = pos + K
            sj = [0] * S
            for r in win:
                if F[r] and c[r] < S:
                    sj[c[r]] = u[r]
            if resolve == "lists":
                resolve_window_lists(a, base, i_cur, sj, rng)
                i_cur -= S
                pos = newpos
                continue
            # ---- swap phase -------------------------------------------------------------------
            own = [a[base + i_cur - s] for s in range(S)]
            flags = [False] * S
            table = {}  # key -> [owner step, value, dup]
            order = list(range(S))
            rng.shuffle(order)  # arbitrary thread interleaving for the CAS race
            for s in order:
                j = sj[s]
                if j > i_cur - S:
                    s2 = i_cur - j
                    if s2 != s:
                        flags[s] = True
                        flags[s2] = True
                else:
                    if j not in table:
                        table[j] = [s, a[base + j], False]
                    else:
                        table[j][2] = True
                        flags[s] = True
            for j, (s_own, _, dup) in table.items():
                if dup:
                    flags[s_own] = True
            # parallel part
            for s in order:
                j = sj[s]
                if flags[s] or j > i_cur - S:
                    continue
                own[s], table[j][1] = table[j][1], own[s]
            # serial part (ascending s)
            nconf = 0
            for s in range(S):
                if not flags[s]:
                    continue
                nconf += 1
                j = sj[s]
                if j > i_cur - S:
                    s2 = i_cur - j
                    own[s], own[s2] = own[s2], own[s]
                else:
                    own[s], table[j][1] = table[j][1], own[s]
            if stats is not None:
                stats["conf"] = stats.get("conf", 0) + nconf
                stats["steps"] = stats.get("steps", 0) + S
            for s in range(S):
                a[base + i_cur - s] = own[s]
            for j, (_, v, _) in table.items():
                a[base + j] = v
            i_cur -= S
            pos = newpos
    return a


def emu_targets(state, inc, segs, Q=4, shortcut="candidates", stats=None):
    """Python emulation of nhood_jgen_kernel (one warp = one generator, 64*Q raw 32-bit values per batch): returns
    {(segment base, i): j}, the Fisher-Yates target of every step, as the kernel streams them to J.

    The window is the rest of the batch capped at i/4.  `shortcut`:
      "candidates"  one pass when no CANDIDATE (u <= i_cur) lies above i_cur - K (what the kernel does);
      "flags"       the same test on the CURRENT flags inside the loop — the first, wrong version of the shortcut (a value
                    rejected in one round can come back in the next), kept so that the test proves it can tell them apart;
      None          always iterate to the fixed point."""
    RAW = 64 * Q
    lanes = 32
    Mn, Cn = _jump_consts(lanes)
    st = []
    for t in range(lanes):
        Mt, Ct = _jump_consts(t + 1)
        st.append((Mt * state + Ct * inc) & M128)
    raw = [0] * RAW
    pos = RAW
    out = {}

    def gen():
        nonlocal pos
        for q in range(Q):
            for t in range(lanes):
                o = _out(st[t])
                raw[q * 64 + 2 * t] = o & 0xFFFFFFFF
                raw[q * 64 + 2 * t + 1] = o >> 32
                st[t] = (Mn * st[t] + Cn * inc) & M128
        pos = 0

    for (base, m) in segs:
        i_cur = m - 1
        while i_cur >= 1:
            if pos >= RAW:
                gen()
            mask = (1 << i_cur.bit_length()) - 1
            i_lo = (mask >> 1) + 1
            n_ph = i_cur - i_lo + 1
            K = min(i_cur >> 2, RAW)
            K = min(max(K, 1), RAW - pos)
            win = list(range(pos, pos + K))
            u = {r: raw[r] & mask for r in win}
            F = {r: u[r] <= i_cur for r in win}  # optimistic start: every candidate accepted
            any_unc = any(F[r] and u[r] > i_cur - K for r in win)
            c = {}
            rounds = 0
            while True:
                rounds += 1
                run = 0
                for r in win:
                    c[r] = run
                    run += 1 if F[r] else 0
                total = run
                if shortcut == "candidates" and not any_unc:
                    break
                if shortcut == "flags" and not any(F[r] and u[r] > i_cur - K for r in win):
                    break
                F2 = {r: (u[r] <= i_cur) and (u[r] <= i_cur - c[r]) for r in win}
                if F2 == F:
                    break
                F = F2
            if stats is not None:
                stats["windows"] = stats.get("windows", 0) + 1
                stats["rounds"] = stats.get("rounds", 0) + rounds
                stats["one_pass"] = stats.get("one_pass", 0) + (1 if rounds == 1 else 0)
            if total >= n_ph:
                S = n_ph
                rstar = next(r for r in win if F[r] and c[r] == S - 1)
                newpos = rstar + 1
            else:
                S = total
                newpos = pos + K
            for r in win:
                if F[r] and c[r] < S:
                    out[(base, i_cur - c[r])] = u[r]
            i_cur -= S
            pos = newpos
    return out


def serial_targets(state, inc, segs):
    """numpy's Generator.shuffle target sequence by plain serial replay: PCG64 next32 (low half first) + masked rejection."""
    s = state
    buf = None
    out = {}

    def next32():
        nonlocal s, buf
        if buf is not None:
            v, buf = buf, None
            return v
        s = (s * A + inc) & M128
        o = _out(s)
        buf = o >> 32
        return o & 0xFFFFFFFF

    for (base, m) in segs:
        for i in range(m - 1, 0, -1):
            mask = (1 << i.bit_length()) - 1
            while True:
                v = next32() & mask
                if v <= i:
                    break
            out[(base, i)] = v
    return out


# ------------------------------------------------------------------------------------------------
# Region replay: executable specification of nhood_apply_region_kernel (shuffle_algo 8, last present in commit eef2f18)
# ------------------------------------------------------------------------------------------------
def _resolve_general_window(slab, a, lo, hi, tops, tgts, rng):
    """One window of the region replay: compacted steps in step order (slot s: top position tops[s], strictly descending;
    target tgts[s] inside the region [lo, hi)).  A top lies above the region (its value T is read from / its final value is
    written to `a`) or inside it (slab).  Every step derives what it writes from per-POSITION lists and original values only:
      targeters[p] = steps with target p (and top != p), owner[p] = the step whose top is p (if it is in this window);
      T(x) = value of x's top just before step x = T(latest targeter of that top) or its original value;
      step s writes  top_s <- value of its target just before s = T(latest earlier targeter of it) or the original;
      the last targeter of p deposits T(itself) at p unless p's owner is in the window (the owner then overwrites p anyway and
      has taken the deposit through T)."""
    S = len(tops)
    otop = [a[tops[s]] if tops[s] >= hi else slab[tops[s] - lo] for s in range(S)]
    targeters, owner = {}, {}
    order = list(range(S))
    rng.shuffle(order)
    for s in order:
        if tops[s] < hi:
            owner[tops[s]] = s
        if tgts[s] != tops[s]:
            targeters.setdefault(tgts[s], []).append(s)
    orig = {p: slab[p - lo] for p in targeters}

    def T(x):
        while targeters.get(tops[x]):
            x = max(targeters[tops[x]])
        return otop[x]

    wa, ws = [], []
    for s in order:
        top, p = tops[s], tgts[s]
        if p == top:
            val = T(s)
        else:
            lst = targeters[p]
            c = [e for e in lst if e < s]
            val = T(max(c)) if c else orig[p]
            if s == max(lst) and p not in owner:
                ws.append((p - lo, T(s)))
        if top >= hi:
            wa.append((top, val))
        else:
            ws.append((top - lo, val))
    for pos, v in wa:
        a[pos] = v
    for pos, v in ws:
        slab[pos] = v


def region_replay(arr, J, cap, NT=8, WL=4, CAPW=12, KMAX=16, rng=None, stats=None):
    """Applies the Fisher-Yates steps i = m-1 .. 1 (swap positions i and J[i] <= i) to a copy of `arr`, one region of at most
    `cap` positions at a time, top region first (see DESIGN.md 3.1): the pass of region [lo, hi) scans all steps i >= lo and
    applies those whose TARGET lies in the region (a step whose target lies below is left to a later pass: its top then
    still holds T(step), the value it had just before the step).  Mirrors the kernel's chunking: NT*K steps are scanned per
    window, "warp" w (WL lanes) takes the w-th run of WL*K of them; K is sized for ~0.58 CAPW expected matches per warp and
    halved when a warp finds more than CAPW or the window more than HS = 2*NT."""
    rng = rng or random.Random(0)
    a = list(arr)
    m = len(a)
    if m < 2:
        return a
    HS = 2 * NT
    ETGT = max(1, (CAPW * 56) // 96)
    assert 2 * WL <= CAPW
    R = (m + cap - 1) // cap
    B = (((m + R - 1) // R + 15) // 16) * 16
    for r in range((m - 1) // B, -1, -1):
        lo = r * B
        ln = min(B, m - lo)
        hi = lo + ln
        slab = a[lo:hi]
        i_min = max(lo, 1)
        i_cur = m - 1
        while i_cur >= i_min:
            avail = i_cur - i_min + 1
            K = min(KMAX, max(2, (ETGT * (i_cur + 1)) // (WL * min(ln, i_cur - lo + 1))))
            while True:
                SC = min(NT * K, avail)
                match = [lo <= J[i_cur - s] < hi for s in range(SC)]
                per_warp = [sum(match[w * WL * K:(w + 1) * WL * K]) for w in range(NT // WL)]
                if max(per_warp) <= CAPW and sum(per_warp) <= HS:
                    break
                K = max(2, K >> 1)
                if stats is not None:
                    stats["overflow"] = stats.get("overflow", 0) + 1
            steps = [i_cur - s for s in range(SC) if match[s]]
            _resolve_general_window(slab, a, lo, hi, steps, [J[i] for i in steps], rng)
            if stats is not None:
                stats["xwin"] = stats.get("xwin", 0) + 1
            i_cur -= SC
        a[lo:hi] = slab
    return a
