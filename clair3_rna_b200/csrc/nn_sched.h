// Launch plan of one network pass's recurrent layers (pure host code: no CUDA, so tests build it with the host
// compiler alone).
//
// A work item of LSTM1 (k_lstm_tc) and of LSTM2 (k_lstm2_fused) is one 256-site tile pair in both directions on
// one "slot" of 4 SMs (a 2-CTA cluster per direction, one CTA per SM).  A pass of P tile pairs on S = sm_count / 4
// slots, run as rounds (LSTM1 of every pair, then LSTM2 of every pair), leaves S - P % S slots idle for a whole
// LSTM1 round and a whole LSTM2 round when P % S != 0.  The two-group plan runs the pass on two disjoint groups
// of slots on two streams instead:
//   group X (sx slots, caller's stream): LSTM1 of pairs [0, sx), LSTM2 of them, then LSTM2 of pairs [sx + ny, P)
//   group Y (sy = S - sx slots, second stream): LSTM1 of pairs [sx, P) in waves, then LSTM2 of [sx, sx + ny)
// so the second group's LSTM1 waves run beside the first group's LSTM2.  L4 + heads (k_gemm_tc, k_l4_finish,
// k_heads_out) of the LSTM2 launch that ends last follow it on its stream; those of every other range go on the
// other stream once its LSTM2 has ended, onto the SMs it released.  The plan is chosen with a slot-level time
// model; the rounds plan is always a candidate and a two-group plan is taken only when the model says it is
// strictly shorter.
#pragma once

namespace c3r {

// Item times of the model, in us: NVIDIA B200 at its 1000 W limit, config 2 (14 617 sites = 58 tile pairs), C = 18.
// k_lstm_tc took 288 us for two rounds; k_lstm2_fused took 383 us for a full round of 37 pairs and 347 us for a
// round of 21; L4 + heads of 21 pairs took ~100 us after the last LSTM2 launch.  Only their ratios matter
// (LSTM2 : LSTM1 = 2.5).
constexpr int SCHED_T_LSTM1 = 144;
constexpr int SCHED_T_LSTM2 = 365;
constexpr int SCHED_T_TAIL = 100;      // per round (S pairs or fewer) of L4 + heads after the LSTM2 they read

enum SchedKind { SCHED_LSTM1 = 0, SCHED_LSTM2 = 1, SCHED_L4H = 2 };

struct SchedLaunch {
    int stream;          // 0 = the caller's stream, 1 = the second stream
    int kind;            // SchedKind
    int p0, np;          // tile pairs [p0, p0 + np)
    int cap;             // at most this many tile pairs at once (slots); 0 for L4 + heads
    int wait;            // index of an earlier launch on the other stream that must end first, or -1
};

struct SchedPlan {
    int n = 0;
    SchedLaunch l[8];
    int split = 0;       // 1: the two-group plan
    int t_model = 0;     // modelled time of the pass (us)
};

inline int sched_ceil(int a, int b) { return (a + b - 1) / b; }
inline int sched_max(int a, int b) { return a > b ? a : b; }

inline void sched_add(SchedPlan& p, int stream, int kind, int p0, int np, int cap, int wait) {
    SchedLaunch& l = p.l[p.n++];
    l.stream = stream; l.kind = kind; l.p0 = p0; l.np = np; l.cap = cap; l.wait = wait;
}

// Today's rounds: LSTM1 of every pair on up to S slots; LSTM2 as A (whole rounds of lstm2_round pairs) and B (the
// rest), with L4 + heads of A on the second stream beside B.
inline SchedPlan sched_rounds(int P, int S, int lstm2_round) {
    SchedPlan p;
    const int pa = P > lstm2_round && P % lstm2_round != 0 ? (P / lstm2_round) * lstm2_round : P;
    sched_add(p, 0, SCHED_LSTM1, 0, P, S, -1);
    sched_add(p, 0, SCHED_LSTM2, 0, pa, lstm2_round, -1);
    const int t_a = sched_ceil(P, S) * SCHED_T_LSTM1 + sched_ceil(pa, lstm2_round) * SCHED_T_LSTM2;
    if (pa == P) {
        sched_add(p, 0, SCHED_L4H, 0, P, 0, -1);
        p.t_model = t_a + sched_ceil(P, S) * SCHED_T_TAIL;
        return p;
    }
    sched_add(p, 0, SCHED_LSTM2, pa, P - pa, lstm2_round, -1);
    sched_add(p, 1, SCHED_L4H, 0, pa, 0, 1);
    sched_add(p, 0, SCHED_L4H, pa, P - pa, 0, -1);
    p.t_model = sched_max(t_a + sched_ceil(pa, S) * SCHED_T_TAIL, t_a + SCHED_T_LSTM2 + sched_ceil(P - pa, S) * SCHED_T_TAIL);
    return p;
}

// Modelled end of the two-group plan with sx slots in group X and ny pairs of LSTM2 in group Y (see the top), or
// -1 when X has LSTM2 pairs of Y's (n2 > 0) and does not end last.  *x_last: X's last LSTM2 launch ends last.
inline int sched_two_group_time(int P, int S, int sx, int ny, int* x_last) {
    const int sy = S - sx, n2 = P - sx - ny;
    const int ty1 = sched_ceil(P - sx, sy) * SCHED_T_LSTM1;                         // Y: LSTM1 of [sx, P)
    const int ty2 = ty1 + (ny ? sched_ceil(ny, sy) * SCHED_T_LSTM2 : 0);             // Y: LSTM2 of [sx, sx + ny)
    const int tx1 = SCHED_T_LSTM1 + SCHED_T_LSTM2;                                   // X: LSTM1 + LSTM2 of [0, sx)
    const int tx2 = n2 ? sched_max(tx1, ty1) + sched_ceil(n2, sx) * SCHED_T_LSTM2 : tx1;   // X: LSTM2 of [sx + ny, P)
    *x_last = tx2 >= ty2;
    if (n2 == 0)                                        // two independent groups, each with its own tail
        return sched_max(tx1 + sched_ceil(sx, S) * SCHED_T_TAIL, ty2 + sched_ceil(ny, S) * SCHED_T_TAIL);
    if (!*x_last) return -1;
    // tails: [0, sx + ny) on Y's slots once Y has ended, [sx + ny, P) after X
    return sched_max(sched_max(ty2, tx1) + sched_ceil(sx + ny, S) * SCHED_T_TAIL, tx2 + sched_ceil(n2, S) * SCHED_T_TAIL);
}

// The plan of a pass of P tile pairs on S slots, LSTM2 taking lstm2_round pairs per round in clusters of
// lstm2_np pairs.  The two-group plan is considered for LSTM2 clusters of one pair (its groups are any number of
// slots) and a partly filled last round (P > S, P % S != 0); otherwise, and when it is not strictly shorter in the
// model, the rounds plan is returned.  Launches are listed in an order they can be issued in, and the LSTM2
// launch listed last is the one that ends last.
inline SchedPlan sched_plan(int P, int S, int lstm2_round, int lstm2_np) {
    SchedPlan best = sched_rounds(P, S, lstm2_round);
    if (lstm2_np != 1 || lstm2_round != S || S < 2 || P <= S || P % S == 0) return best;
    int bt = best.t_model, bsx = 0, bny = 0, bx = 0;
    for (int sx = 1; sx < S; ++sx)
        for (int ny = 0; ny <= P - sx; ++ny) {
            int x_last = 0;
            const int t = sched_two_group_time(P, S, sx, ny, &x_last);
            if (t >= 0 && t < bt) { bt = t; bsx = sx; bny = ny; bx = x_last; }
        }
    if (bsx == 0) return best;
    const int sx = bsx, sy = S - sx, ny = bny, n2 = P - sx - ny;
    SchedPlan p;
    p.split = 1;
    p.t_model = bt;
    sched_add(p, 0, SCHED_LSTM1, 0, sx, sx, -1);                  // 0: X
    sched_add(p, 1, SCHED_LSTM1, sx, P - sx, sy, -1);             // 1: Y, in waves
    if (n2 > 0) {
        sched_add(p, 0, SCHED_LSTM2, 0, sx, sx, -1);              // 2
        if (ny) sched_add(p, 1, SCHED_LSTM2, sx, ny, sy, -1);
        sched_add(p, 0, SCHED_LSTM2, sx + ny, n2, sx, 1);         // its pairs' LSTM1 ran in Y
        sched_add(p, 1, SCHED_L4H, 0, sx + ny, 0, 2);
        sched_add(p, 0, SCHED_L4H, sx + ny, n2, 0, -1);
    } else if (bx) {
        sched_add(p, 1, SCHED_LSTM2, sx, ny, sy, -1);
        sched_add(p, 0, SCHED_LSTM2, 0, sx, sx, -1);
        sched_add(p, 1, SCHED_L4H, sx, ny, 0, -1);
        sched_add(p, 0, SCHED_L4H, 0, sx, 0, -1);
    } else {
        sched_add(p, 0, SCHED_LSTM2, 0, sx, sx, -1);
        sched_add(p, 1, SCHED_LSTM2, sx, ny, sy, -1);
        sched_add(p, 0, SCHED_L4H, 0, sx, 0, -1);
        sched_add(p, 1, SCHED_L4H, sx, ny, 0, -1);
    }
    return p;
}

}  // namespace c3r
