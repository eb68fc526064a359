"""The deque statistics of the five meter columns (csrc/stats_kernel.cuh: stats_kernel, its carried variant and
stats_push1_kernel, through omega4_meter_stats) on hand-built float64 ``lufs_inst`` / ``tp_db`` series, against
``oracle.oracle_np.OracleMeterStats`` pushed with the same doubles.

The series are built where sliding windows with exact order statistics go wrong: plateaus and ties (a duplicate
value expires every hop), monotone runs (every insert at one end of the sorted array), a gated set of 0, 1 and 2
members, values at and within float32 rounding of the gate (which the reference keeps or drops on the double),
mixed signs, the true-peak maximum expiring, every shape of a 32-hop slice and of the 3600 window, and every way
of cutting a series into carried calls.

Tolerance 5e-5 LU on all five columns: inputs and outputs are rounded to float32 (<= 7.6e-6 near 100 LU), while one
wrong gate membership, rank or expiry moves I, LRA or TP by far more.  Carried calls are bit-identical to one call:
every sum adds and subtracts the same float32-rounded values, and those sums are exact."""
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

from oracle import oracle_np as O

pytestmark = pytest.mark.gpu

TOL = 5e-5
INIT = np.array([-100.0, -100.0, -100.0, 0.0, -100.0])      # a fresh meter's outputs before its first push
N_SAT = 7300                                                # saturates the 3600 window twice


def oracle_rows(li, tp, gate=-70.0, first_frame=0):
    """[n, 5] outputs of OracleMeterStats(gate) pushed with li[k], tp[k] for k >= first_frame (INIT before)."""
    st = O.OracleMeterStats()
    st.gate = gate
    out = np.tile(INIT, (len(li), 1))
    for k, (a, b) in enumerate(zip(np.asarray(li).tolist(), np.asarray(tp).tolist())):
        if k >= first_frame:
            d = st.push(a, b)
            out[k] = [d[key] for key in O.METER_KEYS]
    return out


def tp_pattern(n, seed):
    """Peaks with ties of the maximum (a few integer levels), then descending saw-tooth runs in which the maximum
    expires at every hop and the window is rescanned."""
    rng = np.random.default_rng(seed)
    h = n // 2
    tp = np.empty(n)
    tp[:h] = rng.choice([-30.0, -12.0, -6.0, -3.0], h)
    k = np.arange(n - h)
    tp[h:] = -3.0 - 0.015625 * (k % 200)
    return tp


def gate_edges(g, d):
    """Values at, just above and just below the gate g: the double and float32 neighbours of g, and g +- k d."""
    g32 = np.float32(g)
    return np.array([g, np.nextafter(g, 0.0), np.nextafter(g, -np.inf)]
                    + [g + k * d for k in range(1, 9)] + [g - k * d for k in range(1, 4)]
                    + [float(g32), float(np.nextafter(g32, np.float32(0))), float(np.nextafter(g32, np.float32(-np.inf)))])


def edge_series(g, d, n, seed):
    """A loud -20 LUFS at every even hop, the gate-edge values (shuffled cycles) at every odd hop: a wrong
    membership of the edge values moves I by up to 25 LU."""
    rng = np.random.default_rng(seed)
    e = gate_edges(g, d)
    cyc = np.concatenate([rng.permutation(e) for _ in range(n // (2 * len(e)) + 1)])
    li = np.full(n, -20.0)
    li[1::2] = cyc[:len(li[1::2])]
    return li


def ramps(n):
    """Triangle runs of different slopes crossing the gate: up -95 -> -5 over 1000 hops, down over 1500, up over
    333, down over 4000, ..."""
    parts, i = [], 0
    lens = [1000, 1500, 333, 4000, 31, 2900, 64]
    while sum(len(p) for p in parts) < n:
        L = lens[i % len(lens)]
        r = np.linspace(-95.0, -5.0, L)
        parts.append(r if i % 2 == 0 else r[::-1])
        i += 1
    return np.concatenate(parts)[:n]


def mixed(n, seed):
    """Mixed signs and magnitudes: positive LUFS up to +12, values near 0 (|v| >= 0.01, so the float32 sums stay
    exact), 0.0 and the -100 silence value."""
    rng = np.random.default_rng(seed)
    pick = rng.integers(0, 4, n)
    return np.where(pick == 0, rng.uniform(-3.0, 12.0, n),
                    np.where(pick == 1, rng.choice([-1.0, 1.0], n) * rng.uniform(0.01, 0.5, n),
                             np.where(pick == 2, 0.0, -100.0)))


def count_series():
    """Silence except two members: the gated count goes 0 -> 1 (hop 10) -> 2 (hop 20) -> 1 (hop 3610) -> 0 (hop 3620),
    then 1 again (hop 3650) -> 0 (hop 7250)."""
    li = np.full(7300, -100.0)
    li[10], li[20], li[3650] = -30.0, -40.0, -25.0
    return li


def tp_window_series():
    """True peak: the maximum (-5) at hops 10 and 40 expires at hop 70 while its tie is still inside; at hop 100 the
    tie expires into a rescan (-50); then a descending run where the maximum expires at every hop."""
    tp = np.full(400, -50.0)
    tp[10] = tp[40] = -5.0
    tp[200:300] = -10.0 - 0.125 * np.arange(100)
    return tp


GATES = {"edges-70": (-70.0, 1e-6), "edges-70.3": (-70.3, 5e-7), "edges-60": (-60.0, 1e-6), "edges-100": (-100.0, 1e-6)}


def build_series():
    """name -> (lufs_inst, tp_db, gate) for the one-shot comparisons (each saturates the 3600 window twice)."""
    n = N_SAT
    rng = np.random.default_rng(7)
    s = {
        "plateau": np.full(n, -23.0),
        "alternate": np.where(np.arange(n) % 2 == 1, -20.0, -31.5),
        "levels": rng.choice([-80.0, -45.25, -23.0, -18.5, -71.0], n),
        "ramps": ramps(n),
        "mixed": mixed(n, 8),
        "count": count_series(),
    }
    out = {k: (v, tp_pattern(n, i), -70.0) for i, (k, v) in enumerate(s.items())}
    for i, (k, (g, d)) in enumerate(GATES.items()):
        out[k] = (edge_series(g, d, n, 20 + i), tp_pattern(n, 20 + i), g)
    out["tp-window"] = (np.full(400, -23.0), tp_window_series(), -70.0)
    # 20000 hops for the frame-count sweep: pieces of the others, so every kind of value crosses the cuts
    long_li = np.concatenate([s["levels"][:5000], out["edges-70"][0][:5000], s["ramps"][:5000], s["mixed"][:5000]])
    out["long"] = (long_li, tp_pattern(20000, 99), -70.0)
    return out


SERIES = build_series()
ONE_SHOT = [k for k in SERIES if k != "long"]


def _oracle_job(key):
    li, tp, g = SERIES[key[0]]
    return oracle_rows(li, tp, g, key[1])


@pytest.fixture(scope="module")
def ref():
    """Oracle outputs of every series (and of "count" from frame 3), computed once in parallel worker processes."""
    keys = [(k, 0) for k in SERIES] + [("count", 3)]
    ctx = multiprocessing.get_context("fork")
    with ProcessPoolExecutor(max_workers=min(len(keys), os.cpu_count() or 1), mp_context=ctx) as ex:
        res = list(ex.map(_oracle_job, keys))
    return dict(zip(keys, res))


@pytest.fixture(scope="module")
def plan():
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS
    p = AnalysisPlan(48000, BASELINE_CONFIGS, 512)
    yield p
    p.close()


def stats(plan, li, tp, gate=-70.0, **kw):
    plan.set_gate_threshold(gate)
    try:
        return plan.meter_stats_host(li, tp, **kw)
    finally:
        plan.set_gate_threshold(-70.0)


def worst(got, want, label):
    err = np.abs(np.asarray(got, np.float64) - want).max(axis=tuple(range(want.ndim - 1)))
    assert err.max() <= TOL, f"{label}: worst |GPU - oracle| per column (M, S, I, LRA, TP) = {err}"
    return err


def new_state(n_ch=1):
    from omega4_b200 import _native as N
    return np.zeros((n_ch, N.METER_STATE_DOUBLES))


@pytest.mark.parametrize("name", ONE_SHOT)
def test_one_shot_matches_oracle(ref, plan, name):
    li, tp, g = SERIES[name]
    st = new_state()
    got = stats(plan, li, tp, g, state=st, fresh=True)[0]
    err = worst(got, ref[(name, 0)], name)
    print(f"{name}: worst |GPU - oracle| (M, S, I, LRA, TP) = {err}")
    # the carried window holds the unrounded inputs, oldest first
    n = min(len(li), 3600)
    assert int(st[0, 0]) == n and np.array_equal(st[0, 8:8 + n], li[-n:])


def test_gate_edges_decide_on_the_double(plan, ref):
    """The reference keeps a value in (g, g + half a float32 step) that rounds onto g; -100 stays out at -100."""
    assert (SERIES["edges-100"][0] == -100.0).any()
    for name in GATES:
        li, tp, g = SERIES[name]
        # the series holds values whose membership a float32 comparison would get wrong
        assert ((li > g) != (li.astype(np.float32) > np.float32(g))).any(), name
        got = stats(plan, li, tp, g, fresh=True)[0]
        d = np.abs(got[:, 2].astype(np.float64) - ref[(name, 0)][:, 2]).max()
        assert d <= TOL, f"{name}: integrated loudness off by {d} LU"


def test_gated_count_zero_one_two(plan, ref):
    li, tp, g = SERIES["count"]
    got = stats(plan, li, tp, g, fresh=True)[0]
    worst(got, ref[("count", 0)], "count")
    assert np.all(got[:10, 2] == -100.0) and np.all(got[:10, 3] == 0.0)
    assert np.all(got[10:20, 2] == -30.0) and np.all(got[10:20, 3] == 0.0)           # n = 1
    assert np.all(got[20:3610, 2] == -35.0)                                           # n = 2
    assert np.all(np.abs(got[20:3610, 3] - 0.85 * 10.0) <= TOL)                        # P95 - P10 of {-40, -30}
    assert np.all(got[3610:3620, 2] == -40.0) and np.all(got[3620:3650, 2] == -100.0)
    assert np.all(got[3620:3650, 3] == 0.0) and np.all(got[3650:7250, 2] == -25.0) and np.all(got[7250:, 2] == -100.0)


def test_true_peak_window(plan, ref):
    li, tp, g = SERIES["tp-window"]
    got = stats(plan, li, tp, g, fresh=True)[0]
    worst(got, ref[("tp-window", 0)], "tp-window")
    assert np.all(got[10:100, 4] == -5.0) and np.all(got[100:200, 4] == -50.0)
    assert np.array_equal(got[260:300, 4], tp[201:241].astype(np.float32))          # the maximum expires every hop


@pytest.mark.parametrize("n", [1, 31, 32, 33, 255, 257, 3599, 3600, 3601, 7201, 20000])
def test_frame_counts(ref, plan, n):
    li, tp, g = SERIES["long"]
    got = stats(plan, li[:n], tp[:n], g, fresh=True)[0]
    worst(got, ref[("long", 0)][:n], f"n_frames={n}")


def test_first_frame(plan, ref):
    li, tp, g = SERIES["count"]
    got = stats(plan, li, tp, g, first_frame=3, fresh=True)[0]
    worst(got, ref[("count", 3)], "first_frame=3")
    none = stats(plan, li[:50], tp[:50], g, first_frame=60, fresh=True)[0]
    assert np.array_equal(none, np.tile(INIT, (50, 1)).astype(np.float32))
    # on carried state, a call whose first meter frame lies beyond it repeats the carried outputs and keeps the state
    li, tp, g = SERIES["levels"]
    st = new_state()
    a = stats(plan, li[:4000], tp[:4000], g, state=st, fresh=True)[0]
    keep = st.copy()
    b = stats(plan, li[4000:4100], tp[4000:4100], g, state=st, first_frame=200)[0]
    assert np.array_equal(b, np.tile(a[-1], (100, 1))) and np.array_equal(st, keep)
    c = stats(plan, li[4000:], tp[4000:], g, state=st)[0]
    assert np.array_equal(np.concatenate([a, c]), stats(plan, li, tp, g, fresh=True)[0])


@pytest.mark.parametrize("n_ch", [1, 15, 16, 2049])
def test_channel_counts(ref, plan, n_ch):
    """Channel c walks series c % 4 (4000 hops); more than one wave of CTAs at 2049 channels."""
    names = ["levels", "edges-70", "ramps", "mixed"]
    n = 4000
    li = np.stack([SERIES[names[c % 4]][0][:n] for c in range(n_ch)])
    tp = np.stack([SERIES[names[c % 4]][1][:n] for c in range(n_ch)])
    got = stats(plan, li, tp, fresh=True)
    for c in range(min(n_ch, 4)):
        worst(got[c], ref[(names[c], 0)][:n], f"n_ch={n_ch} channel {c} ({names[c]})")
    for c in range(4, n_ch):
        assert np.array_equal(got[c], got[c % 4]), c


def cut_lengths(cut, n, seed=0):
    if cut == "random":
        rng = np.random.default_rng(seed)
        return list(rng.integers(1, 5000, 64))
    if cut == "mix":                                      # omega4_meter_update-style: tiles and single frames
        return [3590] + [1] * 30 + [3601] + [1] * 5 + [n]
    return [cut]


def run_tiled(plan, li, tp, g, lengths):
    st = new_state()
    parts, pos, i = [], 0, 0
    while pos < len(li):
        t = min(int(lengths[i % len(lengths)]), len(li) - pos)
        parts.append(stats(plan, li[pos:pos + t], tp[pos:pos + t], g, state=st, fresh=(pos == 0))[0])
        pos, i = pos + t, i + 1
    return np.concatenate(parts), st


@pytest.mark.parametrize("cut", [1, 2, 31, 32, 33, 3599, 3600, 3601, "random", "mix"])
@pytest.mark.parametrize("name", ["edges-70", "levels", "ramps"])
def test_carried_calls_are_bit_identical(ref, plan, name, cut):
    """Carried calls (the CARRIED walk with its bitonic rebuild; stats_push1_kernel for single frames) == one call."""
    li, tp, g = SERIES[name]
    st1 = new_state()
    one = stats(plan, li, tp, g, state=st1, fresh=True)[0]
    got, st = run_tiled(plan, li, tp, g, cut_lengths(cut, len(li)))
    assert np.array_equal(got, one), f"{name} cut {cut}: first differing hop {np.argwhere(got != one)[:1]}"
    assert np.array_equal(st, st1)
    worst(got, ref[(name, 0)], f"{name} cut {cut}")


def test_single_frames_through_the_walking_kernel(plan, ref):
    """One frame per carried call through the walking kernel (OMEGA4_STATS_WALK=1) == one call, on the gate edges."""
    li, tp, g = SERIES["edges-70.3"]
    li, tp = li[:3700], tp[:3700]
    one = stats(plan, li, tp, g, fresh=True)[0]
    os.environ["OMEGA4_STATS_WALK"] = "1"
    try:
        got, _ = run_tiled(plan, li, tp, g, [1])
    finally:
        del os.environ["OMEGA4_STATS_WALK"]
    assert np.array_equal(got, one)
    worst(got, ref[("edges-70.3", 0)][:3700], "edges-70.3 walk")


def test_gate_change_between_carried_calls(plan):
    """The carried window keeps the unrounded values, so a later call at another gate rebuilds the gated set the
    reference would hold: pushes at -70, then at -70.3, against an oracle whose gate changes at the same hop."""
    li, tp, _ = SERIES["edges-70.3"]
    li, tp = li[:3700], tp[:3700]
    st = new_state()
    a = stats(plan, li[:3650], tp[:3650], -70.0, state=st, fresh=True)[0]
    b = stats(plan, li[3650:], tp[3650:], -70.3, state=st)[0]
    o = O.OracleMeterStats()
    want = []
    for k, (x, y) in enumerate(zip(li.tolist(), tp.tolist())):
        o.gate = -70.0 if k < 3650 else -70.3
        d = o.push(x, y)
        want.append([d[key] for key in O.METER_KEYS])
    worst(np.concatenate([a, b]), np.array(want), "gate change")
