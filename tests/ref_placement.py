"""Plain numpy restatement of place.cu (test infrastructure): the placement of given round counts into rounds, the
round ordering, the fallback priority sweep with its back-off, and the work-conserving back-fill — the same
operation sequence and the same tie-breaking, sequentially.  Used (a) as the reference of that kernel
(tests/test_gpu_placement_ref.py: x and back-fill bit for bit) and (b) to drive the unmodified reference simulator
closed-loop with the product's placement rule on a machine without a GPU (tests/golden/make_placement_pin.py).
The improvement pass of place.cu (idle GPU-rounds handed to jobs below their cap) is not restated: callers only
compare cases in which it does nothing.
"""
import numpy as np


def _waterfill(remn, g, G, Tw, tie):
    """Jobs (descending: all-rounds flag, width, count, tie, index) take their n least-loaded bins that fit.
    Returns (bins[J][Tw] bool, unplaced[J], load[Tw])."""
    J = len(remn)
    xb = np.zeros((J, Tw), dtype=bool)
    left = remn.copy()
    jobs = [j for j in range(J) if remn[j] > 0]
    jobs.sort(key=lambda j: (-(1 if remn[j] >= Tw else 0), -int(g[j]), -int(remn[j]), -int(tie[j]), j))
    ring = [[0, b] for b in range(Tw)]          # logical order: sorted by load, ties by age
    for j in jobs:
        gj, n = int(g[j]), int(remn[j])
        if ring[n - 1][0] <= G - gj and ring[0][0] + gj >= ring[Tw - 1][0]:
            for p in range(n):                  # fast path: the n least-loaded bins move to the end
                xb[j, ring[p][1]] = True
                ring[p][0] += gj
            ring = ring[n:] + ring[:n]
            left[j] = 0
            continue
        u = sum(1 for v in ring if v[0] <= G - gj)
        m = min(n, u)
        if m > 0:
            for p in range(m):
                xb[j, ring[p][1]] = True
            left[j] = n - m
            if m == Tw:
                for v in ring:
                    v[0] += gj
            else:
                X = [[v[0] + gj, v[1]] for v in ring[:m]]
                Y = ring[m:]
                out, ix, iy = [], 0, 0          # stable merge by load; equal loads keep the unmoved bins first
                while ix < len(X) or iy < len(Y):
                    if iy < len(Y) and (ix >= len(X) or Y[iy][0] <= X[ix][0]):
                        out.append(Y[iy]); iy += 1
                    else:
                        out.append(X[ix]); ix += 1
                ring = out
    load = np.zeros(Tw, dtype=np.int64)
    for v in ring:
        load[v[1]] = v[0]
    return xb, left, load


def place(n, g, G, T, bfkey, fallback=False, w=None):
    """Returns dict(x[J][T] bool, backfill[J][T] bool, shortfall, swept_rounds, sweep_stop, idle[T]); sweep_stop is the
    round the fallback sweep stopped at, swept_rounds what is left of it after the back-off."""
    n = np.asarray(n, dtype=np.int64)
    g = np.asarray(g, dtype=np.int64)
    J = len(n)
    prio = fallback and w is not None
    sweep = np.zeros((J, T), dtype=bool)
    idle = np.zeros(T, dtype=np.int64)
    remn = n.copy()
    t0 = 0
    tie = (8191 - np.arange(J)).astype(np.int64)
    if prio:
        w = np.asarray(w, dtype=np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            dens = np.where(n > 0, w / (n.astype(float) * g.astype(float)), -1.0)
        ordr = np.argsort(-dens, kind="stable")
        rank = np.empty(J, dtype=np.int64)
        rank[ordr] = np.arange(J)
        tie = 8192 - rank
        remr = n.copy()
        dem = int((g * n).sum())
        t0 = T
        for t in range(T):
            tau = T - t
            capleft = G
            stage = 0 if np.any(remr >= tau) else 1
            fail = 0
            inr = np.zeros(J, dtype=bool)
            for _ in range(80):
                if stage == 0:
                    el = [j for j in ordr if remr[j] > 0 and not inr[j] and remr[j] >= tau]
                else:
                    el = [j for j in ordr if remr[j] > 0 and not inr[j] and g[j] <= capleft]
                tot = int(sum(g[j] for j in el))
                if stage == 0 and tot > capleft:
                    fail = 1
                    break
                run = taken = 0
                for j in el:
                    run += int(g[j])
                    if run <= capleft:
                        inr[j] = True
                        remr[j] -= 1
                        taken += int(g[j])
                capleft -= taken
                dem -= taken
                if capleft <= 0:
                    break
                if stage == 0:
                    stage = 1
                    continue
                if tot == 0 or taken == tot:
                    break
            sweep[:, t] = inr
            if not fail:
                idle[t] = capleft
                if dem > G * (tau - 1):
                    fail = 2
            if fail:
                tr = t - 1 if (fail == 1 and t > 0) else t
                remr += sweep[:, tr].astype(np.int64)
                sweep[:, tr] = False
                if fail == 1:
                    sweep[:, t] = False
                t0 = tr
                break
        remn = remr.copy()
    t0_sweep = t0
    att = 0
    while True:
        Tw = T - t0
        xb = np.zeros((J, max(Tw, 0)), dtype=bool)
        left = remn.copy()
        load = np.zeros(max(Tw, 0), dtype=np.int64)
        if Tw > 0:
            xb, left, load = _waterfill(remn, g, G, Tw, tie)
        if t0 == 0 or int(left.sum()) == 0:
            break
        nt0 = (t0_sweep * (3 - att)) // 4 if att < 3 else 0
        back = sweep[:, nt0:t0].sum(axis=1)
        sweep[:, nt0:t0] = False
        remr = remr + back
        remn = remr.copy()
        t0 = nt0
        att += 1
    Tw = T - t0
    x = sweep.copy()
    if Tw > 0:
        # order the packer's rounds: most planned work first (fallback: largest sum of prio_j / n_j)
        score = np.zeros(Tw)
        for b in range(Tw):
            members = np.flatnonzero(xb[:, b])
            # warp-per-bin summation order of the kernel: lane l adds jobs l, l+32, ... then a butterfly reduction
            if prio:
                vals = np.zeros(J); vals[members] = w[members] / n[members].astype(float)
            else:
                vals = np.zeros(J); vals[members] = n[members].astype(float) * g[members].astype(float)
            lanes = np.array([_lane_sum(vals, l) for l in range(32)])
            score[b] = _butterfly(lanes)
        order = sorted(range(Tw), key=lambda b: (-score[b], b))
        for pos, b in enumerate(order):
            x[:, t0 + pos] |= xb[:, b]
            idle[t0 + pos] = G - load[b]
    shortfall = int(left.sum())
    # back-fill: descending key (stable), every round independently
    order_bf = np.argsort(-np.asarray(bfkey, dtype=np.float64), kind="stable")
    bf = np.zeros((J, T), dtype=bool)
    for t in range(T):
        room = int(idle[t])
        for j in order_bf:
            if room <= 0:
                break
            if not x[j, t] and g[j] <= room:
                bf[j, t] = True
                room -= int(g[j])
    return dict(x=x, backfill=bf, shortfall=shortfall, swept_rounds=t0, sweep_stop=t0_sweep, idle=idle)


def _lane_sum(vals, lane):
    acc = 0.0
    for j in range(lane, len(vals), 32):
        acc += vals[j]
    return acc


def _butterfly(v):
    v = np.array(v, dtype=np.float64)
    o = 16
    while o > 0:
        v = v + v[np.arange(32) ^ o]
        o >>= 1
    return float(v[0])
