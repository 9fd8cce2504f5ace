"""Per-robot clocks and on-device resets of the gait stack (go1mpc_gait_stack_tick_clocked_async, go1mpc_gait_stack_reset_async):
one batch holds robots at different points of their episodes.

- clocks all at 0 and no reset: the clocked entry is go1mpc_gait_stack_tick_host_async on the reference's schedule, bit for bit;
- staggered episodes (first resets on every residue mod 5, second resets, stop commands on a robot's own planner period): each
  robot's column, body record and rows equal those of a fresh aligned run fed the robot's inputs from its last reset on -- at 16
  robots (combined body kernel) and 2048 (three-launch body path);
- the servo state after a reset, and the servo stack's joint targets after resets against the fresh shifted run;
- one captured period graph (reset + clocked tick + servo) replayed 30 times = 30 direct periods;
- batch-size changes on one stream; argument refusal with no launch and no write."""
import ctypes

import numpy as np
import pytest

import quadrupedal_loco_b200 as q
from tests.test_gpu_gait_stack import SERVO_SLOTS, Stack, planner_ticks, scripted_inputs
from tests.test_gpu_servo_stack import QH, homing_feet

pytestmark = pytest.mark.gpu

NH = 10
K = 10                                   # servo ticks per 10 ms period
Q0 = np.tile(QH, 4)                      # joint angles a reset robot's servo starts from (the homing pose)


def bits(t):
    """Tensor / array viewed as int64 bit patterns (NaN- and signed-zero-exact comparison)."""
    import torch
    if isinstance(t, torch.Tensor):
        return t.contiguous().view(torch.int64)
    return np.ascontiguousarray(t).view(np.int64)


class Farm:
    """One batch on the clocked entry: stack state, body records, result rows, clocks and (optionally) a servo state."""

    def __init__(self, mpc, B, servo_state=None, stream=None):
        import torch
        dev = torch.device("cuda", 0)
        self.mpc, self.B, self.stream = mpc, B, stream
        col = mpc.gait_stack_default_state(NH)
        self.state = torch.from_numpy(np.repeat(col[:, None], B, axis=1).copy()).to(dev)
        self.body_out = torch.zeros(B, q.body_out_stride(NH), dtype=torch.float64, device=dev)
        self.rows_d = torch.zeros(B, len(SERVO_SLOTS), dtype=torch.float64, device=dev)
        self.clock = torch.zeros(B, dtype=torch.int32, device=dev)
        self.servo = None if servo_state is None else torch.from_numpy(np.ascontiguousarray(servo_state)).to(dev)
        self.q_d = torch.zeros(B, 12 * K, dtype=torch.float64, device=dev)

    def reset(self, flags):
        r = self.mpc.gait_stack_reset_struct(NH, flags, self.clock, self.state, self.body_out, self.servo, Q0)
        self.mpc.gait_stack_reset_async(self.B, r, self.stream)

    def tick(self, sensor, cmd=None, start=None):
        t = self.mpc.gait_stack_tick_clocked_struct(NH, sensor, self.clock, self.state, self.body_out, SERVO_SLOTS, self.rows_d,
                                                    cmd=cmd, start=start)
        self.mpc.gait_stack_tick_clocked_async(self.B, t, self.stream)

    def servo_tick(self, state=None):
        self.mpc.servo_stack_tick(self.B, K, 102, 1.0, self.state if state is None else state, self.servo, self.q_d, stream=self.stream)

    def snapshot(self):
        return [t.clone() for t in (self.state, self.body_out, self.clock) + ((self.servo,) if self.servo is not None else ())]


def servo_columns(oracle, B, seed, jitter):
    """Servo state [69][B]: q = Q0 (+ a per-robot jitter), homing feet with a per-robot offset, filters 0 (or random with jitter)."""
    rng = np.random.Generator(np.random.Philox(seed))
    s = np.zeros((q.SERVO_STATE_ROWS, B))
    s[q.SERVO_ROW_Q:q.SERVO_ROW_Q + 12] = Q0[:, None] + (rng.uniform(-0.05, 0.05, (12, B)) if jitter else 0.0)
    s[q.SERVO_ROW_HOMING:q.SERVO_ROW_HOMING + 12] = homing_feet(oracle)[:, None] + rng.uniform(-0.005, 0.005, (12, B))
    if jitter:
        s[q.SERVO_ROW_LPF:] = rng.uniform(-0.1, 0.1, (q.SERVO_STATE_ROWS - q.SERVO_ROW_LPF, B))
    return s


def test_clocked_aligned_equals_host_schedule(mpc):
    """Clocks at 0, no resets, scripted inputs (idle starts, stop / restart commands, control-off windows), 420 periods: the clocked
    entry and go1mpc_gait_stack_tick_host_async with planner_ticks(k) agree bit for bit in state, body records and every period's
    rows; every clock ends at 420."""
    import torch
    R, T = 8, 420
    sensor, cmd, start = scripted_inputs(T, R, 5)
    ref = Stack(mpc, NH, R, SERVO_SLOTS)
    f = Farm(mpc, R)
    rows_ref = torch.zeros(T, R, len(SERVO_SLOTS), dtype=torch.float64, device="cuda")
    rows_f = torch.zeros_like(rows_ref)
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        for k in range(T):
            c, s = np.ascontiguousarray(cmd[k]), np.ascontiguousarray(start[k])
            ref.tick(planner_ticks(k), sensor[k], cmd=c, start=s)
            rows_ref[k].copy_(ref.rows_d)
            f.tick(np.ascontiguousarray(sensor[k]), cmd=c, start=s)
            rows_f[k].copy_(f.rows_d)
    mpc.synchronize(); torch.cuda.synchronize()
    assert torch.equal(bits(f.state), bits(ref.state))
    assert torch.equal(bits(f.body_out), bits(ref.body_out))
    assert torch.equal(bits(rows_f), bits(rows_ref))
    assert (f.clock.cpu().numpy() == T).all()
    assert (np.abs(ref.state[q.STACK_ROW_TRAJ + 72:q.STACK_ROW_TRAJ + 86].cpu().numpy()).sum(axis=0) > 0).sum() >= 6


def reset_schedule(R):
    """Reset periods per robot: first resets at 0..14 (every residue mod 5), every fourth robot reset a second time 31..33 periods
    later, every seventh never reset (its episode starts with the batch)."""
    sched = []
    for r in range(R):
        if r % 7 == 6:
            sched.append([])
            continue
        p1 = r % 5 + 5 * ((r // 5) % 3)
        sched.append([p1] + ([p1 + 31 + r % 3] if r % 4 == 1 else []))
    return sched


E_STOP, E_NOSTOP, E_RESTART = 150, 151, 200      # episode periods: planner, not a planner period, planner


def staggered_inputs(R, T, seed):
    """Staggered-frame inputs [T][..][R], reset flags [T][R], each robot's last reset, and the fresh aligned run's inputs (robot r's
    inputs from its last reset on)."""
    assert planner_ticks(E_STOP) and not planner_ticks(E_NOSTOP) and planner_ticks(E_RESTART)
    sched = reset_schedule(R)
    last = np.array([s[-1] if s else 0 for s in sched])
    flags = np.zeros((T, R), np.int32)
    for r, s in enumerate(sched):
        flags[s, r] = 1
    sensor, _, _ = scripted_inputs(T, R, seed)
    start = np.ones((T, R), np.int32)
    cmd = np.zeros((T, R), np.int32)
    for r in range(R):
        p = last[r]
        start[p:p + 3 * (r % 4), r] = 0                                # idle first periods of the final episode
        events = []
        if r % 6 == 3:
            events.append((E_STOP, 1))                                 # stop, delivered on a planner period of the robot
            if r % 12 == 3:
                events.append((E_RESTART, 2))                          # and walk again
        if r % 6 == 0:
            events.append((E_NOSTOP, 1))                               # not a planner period of the robot: never read
        for e, c in events:
            if p + e < T:
                cmd[p + e, r] = c
    j = np.arange(T)[:, None] + last[None, :]
    jc = np.minimum(j, T - 1)
    cols = np.arange(R)[None, :]
    ref_sensor = sensor.transpose(0, 2, 1)[jc, cols].transpose(0, 2, 1).copy()
    ref_cmd, ref_start = cmd[jc, cols].copy(), start[jc, cols].copy()
    ref_cmd[j >= T] = 0
    return dict(sched=sched, last=last, flags=flags, sensor=sensor, cmd=cmd, start=start, ref_sensor=ref_sensor, ref_cmd=ref_cmd,
                ref_start=ref_start)


def run_staggered(mpc, R, T, seed, servo0=None, ref_servo0=None):
    """The staggered farm (resets + clocked entry [+ servo]) and the fresh aligned run (existing entry [+ servo]) side by side.
    Returns histories of rows (and joint targets) and the full state / body records at two checkpoints, the aligned run's taken at
    each robot's matching episode period."""
    import torch
    dev = torch.device("cuda", 0)
    I = staggered_inputs(R, T, seed)
    last = I["last"]
    f = Farm(mpc, R, servo0)
    ref = Stack(mpc, NH, R, SERVO_SLOTS)
    ref_servo = None if ref_servo0 is None else torch.from_numpy(np.ascontiguousarray(ref_servo0)).to(dev)
    ref_q = torch.zeros(R, 12 * K, dtype=torch.float64, device=dev)
    n = len(SERVO_SLOTS)
    hist = {k: torch.zeros(T, R, n, dtype=torch.float64, device=dev) for k in ("rows", "ref_rows")}
    if servo0 is not None:
        hist.update({k: torch.zeros(T, R, 12 * K, dtype=torch.float64, device=dev) for k in ("q", "ref_q")})
    checks = [T // 2, T - 1]
    snap = {c: None for c in checks}
    ref_snap = {c: [torch.zeros_like(f.state), torch.zeros_like(f.body_out)] for c in checks}
    want_j = {c: c - last for c in checks}                             # the aligned run's period matching checkpoint c, per robot
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        for k in range(T):
            f.reset(np.ascontiguousarray(I["flags"][k]))
            f.tick(np.ascontiguousarray(I["sensor"][k]), cmd=np.ascontiguousarray(I["cmd"][k]), start=np.ascontiguousarray(I["start"][k]))
            hist["rows"][k].copy_(f.rows_d)
            ref.tick(planner_ticks(k), I["ref_sensor"][k], cmd=np.ascontiguousarray(I["ref_cmd"][k]),
                     start=np.ascontiguousarray(I["ref_start"][k]))
            hist["ref_rows"][k].copy_(ref.rows_d)
            if servo0 is not None:
                f.servo_tick()
                hist["q"][k].copy_(f.q_d)
                mpc.servo_stack_tick(R, K, 102, 1.0, ref.state, ref_servo, ref_q)
                hist["ref_q"][k].copy_(ref_q)
            if k in snap:
                snap[k] = [f.state.clone(), f.body_out.clone()]
            for c in checks:
                idx = np.nonzero(want_j[c] == k)[0]
                if idx.size:
                    ix = torch.from_numpy(idx).to(dev)
                    ref_snap[c][0][:, ix] = ref.state[:, ix]
                    ref_snap[c][1][ix] = ref.body_out[ix]
    mpc.synchronize(); torch.cuda.synchronize()
    return I, f, ref, hist, snap, ref_snap


def shifted(hist_ref, last, T):
    """hist_ref[k - last[r], r] for every staggered period k (clamped where k < last[r]) and the mask of k >= last[r]."""
    import torch
    j = torch.arange(T, device=hist_ref.device)[:, None] - torch.from_numpy(last).to(hist_ref.device)[None, :]
    cols = torch.arange(hist_ref.shape[1], device=hist_ref.device)[None, :]
    return hist_ref[j.clamp(min=0), cols], j >= 0


@pytest.mark.parametrize("R", [16, 2048])
def test_staggered_episodes_equal_fresh_shifted_runs(mpc, R):
    """Robots reset at their own periods (first resets on every residue mod 5, some reset twice, resets in periods where other robots
    plan, stop commands on and off a robot's planner periods): each robot's rows at every period of its last episode, and its state
    column and body record at two checkpoints, are bit-identical to a fresh aligned run fed its inputs from its last reset on; its
    clock counts the periods since that reset."""
    import torch
    T = 260
    I, f, ref, hist, snap, ref_snap = run_staggered(mpc, R, T, 61 + R)
    last = I["last"]
    assert set(last % 5) == {0, 1, 2, 3, 4} and any(len(s) == 2 for s in I["sched"])
    # a reset in a period where another robot plans: robot 5 (p = 5) while robot 0 (reset at 0) is at clock 5
    assert 5 in I["sched"][5] and I["sched"][0] == [0] and planner_ticks(5)
    want, live = shifted(hist["ref_rows"], last, T)
    bad = (bits(hist["rows"]) != bits(want)).any(dim=2) & live
    assert bad.sum().item() == 0, f"rows differ for robots {torch.nonzero(bad)[:8, 1].tolist()}"
    for c in snap:
        done = torch.from_numpy(last <= c).to(f.state.device)
        st_bad = ((bits(snap[c][0]) != bits(ref_snap[c][0])).any(dim=0) & done)
        bo_bad = ((bits(snap[c][1]) != bits(ref_snap[c][1])).any(dim=1) & done)
        assert st_bad.sum().item() == 0, f"checkpoint {c}: state columns differ for robots {torch.nonzero(st_bad)[:8, 0].tolist()}"
        assert bo_bad.sum().item() == 0, f"checkpoint {c}: body records differ for robots {torch.nonzero(bo_bad)[:8, 0].tolist()}"
    np.testing.assert_array_equal(f.clock.cpu().numpy(), T - last)
    # the episodes really walked, and the stop command took effect
    S = snap[T - 1][0].cpu().numpy()
    assert (np.abs(S[q.STACK_ROW_TRAJ + 72:q.STACK_ROW_TRAJ + 86]).sum(axis=0) > 0).mean() > 0.5
    assert (S[q.STACK_ROW_NLP + 365, 9::12] != 0).all()                # GO1MPC_NLP_ROW_STOP of the robots that stopped for good


def test_servo_after_reset(mpc, oracle):
    """A reset sets the servo joint angles to servo_q0 and the filter rows to 0, keeps the homing rows and leaves unflagged robots
    untouched; with the servo stack (K = 10) after every period, each robot's joint targets in its last episode equal those of its
    fresh shifted run."""
    import torch
    R = 16
    # (a) what one reset writes, on a batch that has walked and servoed for a few periods
    f = Farm(mpc, R, servo_columns(oracle, R, 3, jitter=True))
    sensor, _, _ = scripted_inputs(8, R, 9)
    torch.cuda.synchronize()
    for k in range(8):
        f.tick(np.ascontiguousarray(sensor[k]))
        f.servo_tick()
    f.body_out.add_(0.5)                                               # every record non-zero before the reset
    mpc.synchronize(); torch.cuda.synchronize()
    before = [t.cpu().numpy() for t in f.snapshot()]
    flags = (np.arange(R) % 3 == 1).astype(np.int32)
    f.reset(flags)
    mpc.synchronize()
    S, BO, C, SV = [t.cpu().numpy() for t in f.snapshot()]
    on, off = flags != 0, flags == 0
    col = mpc.gait_stack_default_state(NH)
    np.testing.assert_array_equal(bits(S[:, on]), bits(np.repeat(col[:, None], on.sum(), axis=1)))
    assert (BO[on] == 0).all() and (C[on] == 0).all()
    np.testing.assert_array_equal(SV[q.SERVO_ROW_Q:q.SERVO_ROW_Q + 12][:, on], np.repeat(Q0[:, None], on.sum(), axis=1))
    np.testing.assert_array_equal(SV[q.SERVO_ROW_HOMING:q.SERVO_ROW_HOMING + 12], before[3][q.SERVO_ROW_HOMING:q.SERVO_ROW_HOMING + 12])
    assert (SV[q.SERVO_ROW_LPF:][:, on] == 0).all()
    np.testing.assert_array_equal(bits(S[:, off]), bits(before[0][:, off]))
    np.testing.assert_array_equal(bits(BO[off]), bits(before[1][off]))
    np.testing.assert_array_equal(C[off], before[2][off])
    np.testing.assert_array_equal(bits(SV[:, off]), bits(before[3][:, off]))
    assert (before[3][q.SERVO_ROW_LPF:][:, on] != 0).any() and (before[2][on] == 8).all()
    # (b) joint targets after staggered resets = the fresh shifted runs'
    T = 230
    fresh = servo_columns(oracle, R, 4, jitter=False)
    start = servo_columns(oracle, R, 4, jitter=True)                   # reset robots start off the fresh column ...
    never = np.array([not s for s in reset_schedule(R)])
    start[:, never] = fresh[:, never]                                   # ... robots never reset start on it
    start[q.SERVO_ROW_HOMING:q.SERVO_ROW_HOMING + 12] = fresh[q.SERVO_ROW_HOMING:q.SERVO_ROW_HOMING + 12]
    I, f, ref, hist, snap, ref_snap = run_staggered(mpc, R, T, 71, servo0=start, ref_servo0=fresh)
    want, live = shifted(hist["ref_q"], I["last"], T)
    bad = (bits(hist["q"]) != bits(want)).any(dim=2) & live
    assert bad.sum().item() == 0, f"joint targets differ for robots {torch.nonzero(bad)[:8, 1].tolist()}"
    assert torch.isfinite(hist["q"]).all() and (hist["q"][-1] != hist["q"][-2]).any()


def test_one_graph_for_every_period(mpc, oracle):
    """After warm-up, one period (reset + clocked tick + servo K = 10) captured once and replayed 30 times -- the pinned sensor and
    reset buffers rewritten between replays, planner and non-planner periods, resets -- equals 30 direct periods bit for bit."""
    import torch
    R, W, N = 64, 6, 30
    s = torch.cuda.Stream()
    sensor, _, _ = scripted_inputs(W + N, R, 83)
    flags = np.zeros((W + N, R), np.int32)
    for r in range(R):
        flags[r % 5, r] = 1                                            # staggered clocks from the warm-up on
        if r % 3 == 0:
            flags[W + 4 + r % 17, r] = 1                               # resets inside the replayed window
    pin_sensor = torch.zeros(q.STACK_SENSOR_ROWS, R, dtype=torch.float64).pin_memory()
    pin_reset = torch.zeros(R, dtype=torch.int32).pin_memory()
    f = Farm(mpc, R, servo_columns(oracle, R, 5, jitter=False), s.cuda_stream)
    hist = {m: (torch.zeros(N, R, len(SERVO_SLOTS), dtype=torch.float64, device="cuda"),
                torch.zeros(N, R, 12 * K, dtype=torch.float64, device="cuda")) for m in ("direct", "graph")}

    def period():
        f.reset(pin_reset)
        f.tick(pin_sensor)
        f.servo_tick()

    def load(k):
        s.synchronize()
        pin_sensor.copy_(torch.from_numpy(sensor[k])); pin_reset.copy_(torch.from_numpy(flags[k]))

    def record(m, j):
        with torch.cuda.stream(s):
            hist[m][0][j].copy_(f.rows_d); hist[m][1][j].copy_(f.q_d)

    torch.cuda.synchronize()
    for k in range(W):
        load(k); period()
    s.synchronize()
    snap0 = f.snapshot()
    for j in range(N):
        load(W + j); period(); record("direct", j)
    s.synchronize()
    want = [t.clone() for t in f.snapshot()]
    for t, t0 in zip((f.state, f.body_out, f.clock, f.servo), snap0):
        t.copy_(t0)
    torch.cuda.synchronize()
    launches = mpc.launch_count
    mpc._check(mpc.lib.go1mpc_graph_capture_begin(mpc.h, s.cuda_stream), "capture_begin")
    period()
    ge = ctypes.c_void_p()
    mpc._check(mpc.lib.go1mpc_graph_capture_end(mpc.h, s.cuda_stream, ctypes.byref(ge)), "capture_end")
    assert mpc.launch_count > launches
    try:
        for j in range(N):
            load(W + j)
            mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, s.cuda_stream), "graph_launch")
            record("graph", j)
        s.synchronize()
    finally:
        mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
    for a, b in zip(hist["graph"], hist["direct"]):
        assert torch.equal(bits(a), bits(b))
    for a, b in zip(f.snapshot(), want):
        assert torch.equal(bits(a) if a.dtype == torch.float64 else a, bits(b) if b.dtype == torch.float64 else b)
    clocks = want[2].cpu().numpy()
    assert len(set(clocks % 5)) == 5 and (clocks < N).any()           # staggered, and resets happened inside the window


def test_batch_size_changes_one_stream(mpc):
    """64 -> 3000 -> 64 robots on one stream, period after period, with both entries: the 64-robot batches equal the first 64 robots
    of the 3000-robot batches given the same inputs (no stale clock mask, reset list or workspace of the larger batch)."""
    import torch
    T, BS, BB = 12, 64, 3000
    s = torch.cuda.Stream()
    sensor, _, _ = scripted_inputs(T, BB, 23)
    flags = np.zeros((T, BB), np.int32)
    for r in range(BB):
        flags[r % 7, r] = 1
    small, big = Farm(mpc, BS, stream=s.cuda_stream), Farm(mpc, BB, stream=s.cuda_stream)
    small_h, big_h = Stack(mpc, NH, BS, SERVO_SLOTS, s.cuda_stream), Stack(mpc, NH, BB, SERVO_SLOTS, s.cuda_stream)
    torch.cuda.synchronize()
    for k in range(T):
        sk = np.ascontiguousarray(sensor[k])
        small.reset(np.ascontiguousarray(flags[k, :BS])); small.tick(np.ascontiguousarray(sk[:, :BS]))
        big.reset(np.ascontiguousarray(flags[k])); big.tick(sk)
        small_h.tick(planner_ticks(k), np.ascontiguousarray(sk[:, :BS])); rs = small_h.rows.copy()
        big_h.tick(planner_ticks(k), sk); rb = big_h.rows.copy()
        s.synchronize()
        assert torch.equal(bits(small.rows_d), bits(big.rows_d[:BS]))
        np.testing.assert_array_equal(rs, rb[:BS])
    torch.cuda.synchronize()
    assert torch.equal(bits(small.state), bits(big.state[:, :BS]))
    assert torch.equal(bits(small.body_out), bits(big.body_out[:BS]))
    assert torch.equal(small.clock, big.clock[:BS])
    assert torch.equal(bits(small_h.state), bits(big_h.state[:, :BS]))


def test_clocked_and_reset_reject_bad_arguments(mpc):
    """Each bad argument returns its code, launches nothing and writes neither state nor clock."""
    import torch
    B = 64
    f = Farm(mpc, B)
    sensor = np.zeros((q.STACK_SENSOR_ROWS, B)); sensor[0] = 1.0
    flags = np.ones(B, np.int32)
    raw = torch.zeros(B * q.body_out_stride(NH) + 2, dtype=torch.float64, device="cuda")
    f.state.add_(1.0)                                                  # not the default column: a stray reset would show
    f.clock.fill_(7)
    tick_ok = dict(nh=NH, sensor=sensor, clock_d=f.clock, state_d=f.state, body_out_d=f.body_out, slots=SERVO_SLOTS, rows_d=f.rows_d)
    reset_ok = dict(nh=NH, reset=flags, clock_d=f.clock, state_d=f.state, body_out_d=f.body_out)

    def tick_rc(B=B, **kw):
        a = dict(tick_ok); a.update(kw)
        return mpc.lib.go1mpc_gait_stack_tick_clocked_async(mpc.h, B, ctypes.byref(mpc.gait_stack_tick_clocked_struct(**a)), None)

    def reset_rc(B=B, **kw):
        a = dict(reset_ok); a.update(kw)
        return mpc.lib.go1mpc_gait_stack_reset_async(mpc.h, B, ctypes.byref(mpc.gait_stack_reset_struct(**a)), None)

    bad_body = raw[1:].data_ptr()
    tick_cases = [
        (dict(clock_d=None), -1), (dict(state_d=None), -1), (dict(body_out_d=None), -1), (dict(sensor=None), -1), (dict(rows_d=None), -1),
        (dict(nh=2), -4), (dict(nh=41), -4), (dict(body_out_d=bad_body), -1),
        (dict(slots=[0, 200]), -1), (dict(slots=[-1]), -1), (dict(slots=[]), -1), (dict(slots=[0] * 65), -1), (dict(B=-1), -1),
    ]
    reset_cases = [
        (dict(reset=None), -1), (dict(clock_d=None), -1), (dict(state_d=None), -1), (dict(body_out_d=None), -1),
        (dict(nh=2), -4), (dict(nh=41), -4), (dict(body_out_d=bad_body), -1), (dict(B=-1), -1),
    ]
    torch.cuda.synchronize()
    state0, clock0 = f.state.clone(), f.clock.clone()
    before = mpc.launch_count
    for kw, code in tick_cases:
        assert tick_rc(**kw) == code, kw
    for kw, code in reset_cases:
        assert reset_rc(**kw) == code, kw
    assert mpc.lib.go1mpc_gait_stack_tick_clocked_async(mpc.h, B, None, None) == -1
    assert mpc.lib.go1mpc_gait_stack_reset_async(mpc.h, B, None, None) == -1
    assert tick_rc(B=0) == 0 and reset_rc(B=0) == 0                    # B = 0: a no-op
    mpc.synchronize(); torch.cuda.synchronize()
    assert mpc.launch_count == before
    assert torch.equal(f.state, state0) and torch.equal(f.clock, clock0)
    # valid calls still work after the refusals
    assert reset_rc() == 0 and tick_rc() == 0
    mpc.synchronize()
    assert mpc.launch_count > before
    assert (f.clock.cpu().numpy() == 1).all()
