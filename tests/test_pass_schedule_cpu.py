"""The pass planner of the tensor-core network (clair3_rna_b200/csrc/nn_sched.h), built with the host compiler.

For P = 1..400 tile pairs on 132, 148 and 160 SMs, every plan is replayed on a slot-level clock that follows the
launch order of tc_forward (stream order, each launch's wait, and the waits tc_forward adds after the last LSTM1 and
the last two LSTM2 launches).  It must run every stage of every pair once and in order, never hold more tile pairs
at once than the SMs take, and never take longer than the rounds schedule."""
import os
import shutil
import subprocess

import pytest

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "clair3_rna_b200", "csrc")
SMS = (132, 148, 160)
MAX_P = 400
L1, L2, L4H = 0, 1, 2

PROGRAM = r"""
#include "nn_sched.h"
#include <cstdio>
static void put(const char* tag, int sm, int P, const c3r::SchedPlan& p) {
    printf("%s %d %d %d %d %d\n", tag, sm, P, p.split, p.t_model, p.n);
    for (int i = 0; i < p.n; ++i)
        printf("%d %d %d %d %d %d\n", p.l[i].stream, p.l[i].kind, p.l[i].p0, p.l[i].np, p.l[i].cap, p.l[i].wait);
}
int main() {
    printf("%d %d %d\n", c3r::SCHED_T_LSTM1, c3r::SCHED_T_LSTM2, c3r::SCHED_T_TAIL);
    const int sms[] = {%SMS%};
    for (int sm : sms)
        for (int P = 1; P <= %MAX_P%; ++P) {
            const int S = sm / 4;
            put("plan", sm, P, c3r::sched_plan(P, S, S, 1));
            put("rounds", sm, P, c3r::sched_rounds(P, S, S));
            put("np2", sm, P, c3r::sched_plan(P, S, (sm / 4 / 2) * 2, 2));
        }
}
"""


@pytest.fixture(scope="module")
def plans(tmp_path_factory):
    cxx = shutil.which("c++") or shutil.which("g++")
    if cxx is None:
        pytest.skip("no host C++ compiler")
    d = tmp_path_factory.mktemp("sched")
    src = d / "plans.cpp"
    src.write_text(PROGRAM.replace("%SMS%", ", ".join(map(str, SMS))).replace("%MAX_P%", str(MAX_P)))
    exe = d / "plans"
    subprocess.run([cxx, "-std=c++17", "-O2", "-Wall", "-Werror", "-I", CSRC, str(src), "-o", str(exe)], check=True)
    lines = subprocess.run([str(exe)], check=True, stdout=subprocess.PIPE, text=True).stdout.splitlines()
    times = tuple(map(int, lines[0].split()))
    out, i = {}, 1
    while i < len(lines):
        tag, sm, P, split, t, n = lines[i].split()
        launches = [tuple(map(int, l.split())) for l in lines[i + 1:i + 1 + int(n)]]
        out[(tag, int(sm), int(P))] = dict(split=int(split), t=int(t), l=launches)
        i += 1 + int(n)
    return times, out


def ceil(a, b):
    return -(-a // b)


def replay(plan, S, times):
    """start / end of every launch on the model's clock, in tc_forward's launch order"""
    t1, t2, tail = times
    ls = plan["l"]
    kinds = [l[1] for l in ls]
    l1_last = max(i for i, k in enumerate(kinds) if k == L1)
    l2 = [i for i, k in enumerate(kinds) if k == L2]
    sync_after = {l1_last: L1, l2[-1]: L2}
    if len(l2) > 1:
        sync_after[l2[-2]] = L2
    free = [0, 0]                    # when each stream's queue is free
    start, end = [], []
    for i, (s, k, p0, np_, cap, w) in enumerate(ls):
        b = max(free[s], end[w] if w >= 0 else 0)
        if w >= 0:
            assert ls[w][0] != s, "a wait names a launch on its own stream"
        dur = ceil(np_, cap) * (t1 if k == L1 else t2) if k != L4H else ceil(np_, S) * tail
        start.append(b)
        end.append(b + dur)
        free[s] = b + dur
        if i in sync_after:          # the stream also waits for the last launch of that kind on the other stream
            j = [q for q in range(i) if ls[q][1] == sync_after[i] and ls[q][0] != s]
            if j:
                free[s] = max(free[s], end[j[-1]])
    return start, end


def check(plan, P, S, times):
    start, end = replay(plan, S, times)
    ls = plan["l"]
    assert len(ls) <= 8
    done = {}
    for i, (s, k, p0, np_, cap, w) in enumerate(ls):
        assert np_ >= 1 and 0 <= p0 and p0 + np_ <= P and s in (0, 1)
        assert (cap >= 1) if k != L4H else cap == 0
        for q in range(p0, p0 + np_):
            assert (k, q) not in done, "pair %d gets stage %d twice" % (q, k)
            if k != L1:
                assert (k - 1, q) in done and start[i] >= end[done[(k - 1, q)]], "pair %d: stage %d before %d" % (q, k, k - 1)
            done[(k, q)] = i
    assert len(done) == 3 * P
    # recurrent launches hold min(np, cap) slots from start to end
    pts = sorted(set(start + end))
    for t in pts:
        held = sum(min(l[3], l[4]) for i, l in enumerate(ls) if l[1] != L4H and start[i] <= t < end[i])
        assert held <= S, "%d slots held at t = %d" % (held, t)
    assert max(end) == plan["t"], "plan's own time %d, replayed %d" % (plan["t"], max(end))
    return max(end)


@pytest.mark.parametrize("sm", SMS)
def test_every_plan_is_complete_fits_and_is_no_slower(plans, sm):
    times, out = plans
    S = sm // 4
    n_split = 0
    for P in range(1, MAX_P + 1):
        rounds = out[("rounds", sm, P)]
        t_r = check(rounds, P, S, times)
        p = out[("plan", sm, P)]
        t = check(p, P, S, times)
        assert t <= t_r, P
        assert p["split"] == (t < t_r), P
        if P <= S or P % S == 0:
            assert p == rounds, P
        n_split += p["split"]
        # LSTM2 clusters of two pairs: always rounds
        p2 = out[("np2", sm, P)]
        check(p2, P, S, times)
        assert p2["split"] == 0, P
    assert n_split > 0


def test_rounds_plan_is_the_launch_list_of_rounds(plans):
    _, out = plans
    # 58 pairs on 148 SMs: LSTM1 of all, LSTM2 of 37 + 21, L4 + heads of the 37 on the second stream
    assert out[("rounds", 148, 58)]["l"] == [(0, L1, 0, 58, 37, -1), (0, L2, 0, 37, 37, -1), (0, L2, 37, 21, 37, -1),
                                             (1, L4H, 0, 37, 0, 1), (0, L4H, 37, 21, 0, -1)]
    assert out[("rounds", 148, 20)]["l"] == [(0, L1, 0, 20, 37, -1), (0, L2, 0, 20, 37, -1), (0, L4H, 0, 20, 0, -1)]


def test_config2_pass_runs_in_two_groups(plans):
    times, out = plans
    p = out[("plan", 148, 58)]
    assert p["split"] == 1
    assert p["t"] < out[("rounds", 148, 58)]["t"]
    caps = {l[4] for l in p["l"] if l[1] == L1}
    assert sum(caps) == 37 and len(caps) == 2
