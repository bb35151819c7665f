"""The segment hand-off protocol of k_trace (torj_jl_b200/csrc/torj_handoff.cuh), checked exhaustively on the CPU.

Under the hand-off a ray's segments are separate work items. They are drawn in queue order but may be claimed in any order,
and the lane that runs a segment hands it in or retires the ray. The per-ray word seg_done changes only through the two
transitions of the header, claim and hand-in, each applied in one compare-and-swap on the device. So the protocol is right
when every interleaving of those transitions for one ray is: the header is compiled with g++ and an explorer walks every
order of claims, hand-ins and retirements.

The explorer is shown to catch the bug it exists for: the earlier transitions (restated below) let two lanes run the same
segment as soon as a ray has 3 segments."""
import ctypes as C
import functools
import os
import subprocess

import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "torj_jl_b200", "csrc")
SHIM = r"""
#include "torj_handoff.cuh"
extern "C" {
int seg_claim(int w, int wseg, int* go) { TorjSegMove m = torj_seg_claim(w, wseg); *go = m.go; return m.w; }
int seg_hand_in(int w, int seg, int* go) { TorjSegMove m = torj_seg_hand_in(w, seg); *go = m.go; return m.w; }
int seg_retired(void) { return TORJ_SEG_RETIRED; }
int seg_max(void) { return TORJ_SEG_MAX; }
}
"""
RETIRED = 0x7FFFFFFF


def done(w):
    return w & 0x7FFF


def drop(w):
    return (w >> 15) & 0x7FFF


class Protocol:
    """The header's transitions through ctypes, memoised (the explorer asks the same questions many times)."""

    def __init__(self, lib):
        self.lib = lib
        for f in (lib.seg_claim, lib.seg_hand_in):
            f.argtypes, f.restype = [C.c_int, C.c_int, C.POINTER(C.c_int)], C.c_int
        self.retired, self.seg_max = lib.seg_retired(), lib.seg_max()

    @functools.lru_cache(maxsize=None)
    def claim(self, w, wseg):
        go = C.c_int(-1)
        nw = self.lib.seg_claim(w, wseg, C.byref(go))
        return nw, bool(go.value)

    @functools.lru_cache(maxsize=None)
    def hand_in(self, w, seg):
        go = C.c_int(-1)
        nw = self.lib.seg_hand_in(w, seg, C.byref(go))
        return nw, bool(go.value)


@pytest.fixture(scope="module")
def proto(tmp_path_factory):
    d = tmp_path_factory.mktemp("handoff")
    src = d / "shim.cpp"
    src.write_text(SHIM)
    so = str(d / "libhandoff.so")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-shared", "-fPIC", "-I" + CSRC, "-o", so,
                           str(src)])
    return Protocol(C.CDLL(so))


# The transitions before the RUNNING bit: a claim was ready whenever DONE == wseg, and the hand-in was one atomicAdd whose
# old value decided whether the lane continued.
def parent_claim(w, wseg):
    if w == RETIRED or done(w) > wseg:
        return w, False
    if done(w) == wseg:
        return w, True
    return done(w) | (max(drop(w), wseg + 1) << 15), False


def parent_hand_in(w, seg):
    return w + 1, drop(w) >= seg + 1


def explore(claim, hand_in, n_seg, first=0):
    """Every interleaving for one ray whose segments first .. n_seg-1 are still to come (the ones before `first` ran
    without drops, so its word starts as DONE = first):
    - each item is claimed exactly once, in any order;
    - a lane that runs segment k hands it in, or retires the ray early (psi / power stop, a fatal status); after the last
      segment it retires;
    - a ready claim of segment 0 may meet a failed initialisation and retire the ray at once.
    Returns (violations, number of states)."""
    m = n_seg - first
    # state: word, unclaimed items, segments being run (a sorted tuple, one entry per lane), runs per segment,
    # last segment before retirement (None: not retired; first - 1: retired before any ran)
    start = (first, frozenset(range(first, n_seg)), (), (0,) * m, None)
    seen, stack, bad = set(), [start], []

    def check(before, after, what):
        if after == RETIRED:
            if before != RETIRED:
                bad.append((what, "a transition made a live word RETIRED", before))
        elif before == RETIRED:
            bad.append((what, "a transition revived a retired word", after))
        elif done(after) > n_seg or drop(after) > n_seg:
            bad.append((what, f"DONE {done(after)} / DROP {drop(after)} beyond {n_seg} segments", after))

    def bump(runs, k):
        r = list(runs)
        r[k - first] += 1
        return tuple(r)

    while stack:
        s = stack.pop()
        if s in seen:
            continue
        seen.add(s)
        w, un, running, runs, end = s
        if not un and not running:
            # nothing can happen any more: the ray must have retired, after each segment up to retirement ran once
            if w != RETIRED:
                bad.append(("stuck", "all items claimed, no lane runs, the ray is not retired", s))
            elif runs != tuple(1 if first + j <= end else 0 for j in range(m)):
                bad.append(("runs", f"retired after segment {end}", s))
            continue
        for j in un:
            nw, go = claim(w, j)
            check(w, nw, f"claim of segment {j}")
            if w == RETIRED and go:
                bad.append((f"claim of segment {j}", "ready after retirement", s))
            if go:
                stack.append((nw, un - {j}, tuple(sorted(running + (j,))), bump(runs, j), end))
                if j == 0:  # failed initialisation: the lane retires the ray at once
                    stack.append((RETIRED, un - {j}, running, runs, first - 1))
            else:
                stack.append((nw, un - {j}, running, runs, end))
        for i, k in enumerate(running):
            rest = running[:i] + running[i + 1:]
            if end is not None:
                bad.append((f"lane of segment {k}", "runs after the ray retired", s))
                continue
            stack.append((RETIRED, un, rest, runs, k))  # retires after segment k
            if k + 1 < n_seg:
                nw, go = hand_in(w, k + 1)
                check(w, nw, f"hand-in of segment {k}")
                if go:
                    stack.append((nw, un, tuple(sorted(rest + (k + 1,))), bump(runs, k + 1), end))
                else:
                    stack.append((nw, un, rest, runs, end))
    return bad, len(seen)


def test_word_layout(proto):
    assert proto.retired == RETIRED
    # a live word has DONE <= n_segments <= TORJ_SEG_MAX, below the all-ones field that RETIRED carries
    assert proto.seg_max == 16000 and proto.seg_max < 0x7FFF


@pytest.mark.parametrize("n_seg", range(1, 8))
def test_every_segment_runs_exactly_once(proto, n_seg):
    bad, n_states = explore(proto.claim, proto.hand_in, n_seg)
    assert not bad, bad[:5]
    assert n_states > 2 * n_seg


def test_top_of_the_segment_range(proto):
    """The last 7 segments of a 16 000-segment ray: the same exhaustive check with DONE and DROP near their limit, and no
    transition from a word near the limit yields RETIRED or a field beyond n_segments."""
    n = proto.seg_max
    bad, _ = explore(proto.claim, proto.hand_in, n, first=n - 7)
    assert not bad, bad[:5]
    near = list(range(4)) + list(range(n - 4, n + 1))
    for d in near:
        for p in [0] + [x + 1 for x in near if x < n]:
            for run in (0, 1 << 30):
                w = d | (p << 15) | run
                for k in near:
                    if k < n:
                        nw, go = proto.claim(w, k)
                        assert nw != RETIRED and done(nw) <= n and drop(nw) <= n, (w, k, nw)
                        assert not go or (done(w) == k and not run and nw == w | (1 << 30)), (w, k, nw)
                    if d < n and 1 <= k <= n:
                        nw, go = proto.hand_in(w, k)
                        assert nw != RETIRED and done(nw) == d + 1 and bool(nw & (1 << 30)) == go, (w, k, nw)
    for k in (0, 1, n - 1):
        assert proto.claim(RETIRED, k) == (RETIRED, False)


def test_explorer_finds_the_double_run_of_the_parent_transitions():
    """The transitions before the RUNNING bit: two lanes run the same segment of a 3-segment ray when item 2's claim
    overtakes item 1's: it drops item 2, the holder of segment 0 continues with segment 1 on handing in, and the late
    claim of item 1 is also ready. With 4 and more segments a segment can also be skipped."""
    assert explore(parent_claim, parent_hand_in, 2)[0] == []
    bad, _ = explore(parent_claim, parent_hand_in, 3)
    states = [s for _, _, s in bad if isinstance(s, tuple)]
    assert any(max(s[3]) == 2 for s in states), bad[:5]
    bad, _ = explore(parent_claim, parent_hand_in, 4)
    assert any(what == "stuck" and 0 in s[3] for what, _, s in bad), bad[:5]  # the last segment never runs
