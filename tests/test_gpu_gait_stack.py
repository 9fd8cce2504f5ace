"""The gait stack tick (go1mpc_gait_stack_tick_host_async): both MPC nodes behind one host call per 100 Hz tick, sensor rows up,
selected result slots down, every node member and both messages resident in one SoA state.

- the cfg1 golden replay of tests/test_gpu_chain.py through the one call;
- bit for bit the two node entries chained by hand (robots out of phase: idle stretches, stop / restart, control off, random
  body angles and foot feedback routed from /rt2nrt/state back into the planner);
- the oracle chain OracleNlpNode -> OracleRtNode on the CPU with the same feedback;
- the host interface: batch-size changes on one stream, graph capture, argument checks that launch nothing."""
import ctypes

import numpy as np
import pytest

import quadrupedal_loco_b200 as q
from tests.test_oracle_vs_ref import OracleNlpNode, OracleRtNode, load

pytestmark = pytest.mark.gpu

SERVO_SLOTS = [0, 1, 2, 6, 7, 8, 9, 10, 11, 39, 40, 41, 172, 173, 174, 175]   # /MPC/Gait 0-2, 6-11, 39-41; /rtMPC/traj 72-75
CTL_SLOTS = [0, 10, 11, 13, 14, 19, 20, 21, 22, 23, 24]                      # /control2rtmpc/state slot of each sensor row


def planner_ticks(k):
    """The fast tick at 10k ms runs the planner first when a multiple of 25 lies in (10(k-1), 10k]."""
    return k == 0 or (10 * k) // 25 > (10 * (k - 1)) // 25


class Stack:
    """One batch on the gait stack entry: device state, body records, result rows."""

    def __init__(self, mpc, nh, B, slots, stream=None):
        import torch
        dev = torch.device("cuda", 0)
        self.mpc, self.nh, self.B, self.slots, self.stream = mpc, nh, B, list(slots), stream
        col = mpc.gait_stack_default_state(nh)
        self.state = torch.from_numpy(np.repeat(col[:, None], B, axis=1).copy()).to(dev)
        self.body_out = torch.zeros(B, q.body_out_stride(nh), dtype=torch.float64, device=dev)
        self.rows_d = torch.zeros(B, len(self.slots), dtype=torch.float64, device=dev)
        self.rows = np.zeros((B, len(self.slots)))

    def tick(self, planner, sensor, cmd=None, start=None):
        t = self.mpc.gait_stack_tick_struct(self.nh, planner, np.ascontiguousarray(sensor), self.state, self.body_out, self.slots,
                                            self.rows_d, self.rows, cmd=cmd, start=start)
        self.mpc.gait_stack_tick_host_async(self.B, t, self.stream)

    def block(self, row, n):
        return self.state[row:row + n]


def test_gait_stack_golden_replay(mpc):
    """cfg1 (tests/golden/rt_node_ref.npz, nh = 4): the planner every 25 ms, the fast node every 10 ms, control flag 1 and every
    other sensor slot 0 -- every /rtMPC/traj to 1e-8, integer slots exact; the rows are the selected slots exactly."""
    import torch
    g = load("rt_node_ref.npz")
    nh = int(g["nh"][0])
    want, mo = g["out"], g["msg_of_fast"]
    R, T = 4, len(g["out"])
    st = Stack(mpc, nh, R, SERVO_SLOTS + [27, 63, 98, 99, 127, 163, 198, 199])
    sensor = np.zeros((q.STACK_SENSOR_ROWS, R)); sensor[0] = 1.0
    traj = torch.zeros(T, 100, R, dtype=torch.float64, device="cuda")
    gait = torch.zeros(T, 100, R, dtype=torch.float64, device="cuda")
    rows = np.zeros((T, R, len(st.slots)))
    count = 0
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        for k in range(T):
            pl = planner_ticks(k)
            count += pl
            assert mo[k] == count
            st.tick(pl, sensor)                                  # rows come down synchronously (pageable host buffer)
            traj[k].copy_(st.block(q.STACK_ROW_TRAJ, 100)); gait[k].copy_(st.block(q.STACK_ROW_GAIT, 100))
            rows[k] = st.rows
    mpc.synchronize(); torch.cuda.synchronize()
    got = traj.cpu().numpy().transpose(0, 2, 1)
    ints = [27, 63, 98, 99]
    for r in range(R):
        np.testing.assert_array_equal(got[:, r][:, ints], want[:, ints])
        err = np.abs(got[:, r] - want) / np.maximum(1.0, np.abs(want))
        assert np.isfinite(got).all() and err.max() < 1e-8, f"robot {r}: {err.max():.3e}"
    both = np.concatenate([gait.cpu().numpy(), traj.cpu().numpy()], axis=1)          # [T, 200, R]
    np.testing.assert_array_equal(rows, both[:, st.slots].transpose(0, 2, 1))
    assert (np.abs(want[:, 72:86]).sum(axis=1) > 0).sum() > 1500


def scripted_inputs(T, R, seed):
    """Sensor rows [T][11][R], planner cmd / start [T][R]: robots out of phase (idle stretches of different lengths), stop and
    restart commands, control-flag-off windows, random body angles / rates and foot feedback around the nominal stance."""
    rng = np.random.Generator(np.random.Philox(seed))
    T_all, T = T, max(T, 320)                                        # the script's events lie within 320 ticks
    sensor = np.zeros((T, q.STACK_SENSOR_ROWS, R))
    sensor[:, 0] = 1.0
    sensor[:, 1:5] = rng.uniform(-0.03, 0.03, (T, 4, R))
    for base, y in ((5, 0.127), (8, -0.127)):                        # left foot xyz, right foot xyz
        sensor[:, base] = rng.uniform(-0.02, 0.02, (T, R))
        sensor[:, base + 1] = y + rng.uniform(-0.01, 0.01, (T, R))
        sensor[:, base + 2] = rng.uniform(-0.005, 0.005, (T, R))
    for t0, t1, r in ((50, 62, 3), (180, 200, 6), (300, 305, 0)):  # control flag off
        if r < R:
            sensor[t0:t1, 0, r] = 0.0
    start = np.ones((T, R), np.int32)
    for r in range(R):
        start[:12 * r, r] = 0                                        # robot r idles for its first 12 r fast ticks
    cmd = np.zeros((T, R), np.int32)
    # robot 2: stop, then walk again; robot 5: stop for good; robot 7: a start command while walking
    for t, r, c in ((150, 2, 1), (230, 2, 2), (260, 5, 1), (100, 7, 2)):
        if r < R:
            cmd[t, r] = c
    return sensor[:T_all], cmd[:T_all], start[:T_all]


def test_gait_stack_equals_separate_entries(mpc):
    """The stack and go1mpc_nlp_node_tick_batch + go1mpc_rt_node_tick_msgs_batch chained by hand (feedback from the previous
    /rt2nrt/state) agree bit for bit: state blocks, body records, messages, rows."""
    import torch
    nh, R, T = 10, 8, 420
    dev = torch.device("cuda", 0)
    sensor, cmd, start = scripted_inputs(T, R, 5)
    st = Stack(mpc, nh, R, SERVO_SLOTS)
    nlp = torch.from_numpy(np.repeat(mpc.nlp_node_default_state()[:, None], R, axis=1).copy()).to(dev)
    rt = torch.from_numpy(np.repeat(mpc.rt_node_default_state(nh)[:, None], R, axis=1).copy()).to(dev)
    gait = torch.zeros(100, R, dtype=torch.float64, device=dev); traj = torch.zeros_like(gait)
    r2n = torch.zeros(25, R, dtype=torch.float64, device=dev); ctl = torch.zeros_like(r2n)
    body_in = torch.zeros(R, q.body_in_stride(nh), dtype=torch.float64, device=dev)
    body_out = torch.zeros(R, q.body_out_stride(nh), dtype=torch.float64, device=dev)
    wd = torch.zeros(R, dtype=torch.int32, device=dev)
    cmd_d = torch.from_numpy(cmd).to(dev); start_d = torch.from_numpy(start).to(dev)
    sensor_d = torch.from_numpy(sensor).to(dev)
    rows_all = np.zeros((T, R, len(SERVO_SLOTS)))
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        for k in range(T):
            pl = planner_ticks(k)
            st.tick(pl, sensor[k], cmd=np.ascontiguousarray(cmd[k]), start=np.ascontiguousarray(start[k]))
            rows_all[k] = st.rows
            if pl:
                wd += 1
                mpc.nlp_node_tick(R, nlp, wd, gait, start_d=start_d[k], cmd_d=cmd_d[k], rfoot_fb_d=r2n[22:25], lfoot_fb_d=r2n[19:22])
            ctl[CTL_SLOTS] = sensor_d[k]
            mpc.rt_node_tick_msgs(nh, R, rt, gait, ctl, body_in, body_out, traj, r2n)
    mpc.synchronize(); torch.cuda.synchronize()
    S = st.state.cpu().numpy()
    np.testing.assert_array_equal(S[q.STACK_ROW_NLP:q.STACK_ROW_GAIT], nlp.cpu().numpy())
    np.testing.assert_array_equal(S[q.STACK_ROW_GAIT:q.STACK_ROW_RT2NRT], gait.cpu().numpy())
    np.testing.assert_array_equal(S[q.STACK_ROW_RT2NRT:q.STACK_ROW_WALKDTIME], r2n.cpu().numpy())
    np.testing.assert_array_equal(S[q.STACK_ROW_WALKDTIME], wd.cpu().numpy().astype(np.float64))
    np.testing.assert_array_equal(S[q.STACK_ROW_TRAJ:q.STACK_ROW_RT], traj.cpu().numpy())
    np.testing.assert_array_equal(S[q.STACK_ROW_RT:], rt.cpu().numpy())
    np.testing.assert_array_equal(st.body_out.cpu().numpy(), body_out.cpu().numpy())
    both = np.concatenate([gait.cpu().numpy(), traj.cpu().numpy()])
    np.testing.assert_array_equal(rows_all[-1], both[SERVO_SLOTS].T)
    # the script really exercised the nodes: robots walk (body MPC ran), robot 5 stopped, robot 3 lost its control window
    assert (np.abs(traj.cpu().numpy()[72:86]).sum(axis=0) > 0).sum() >= 6
    assert np.unique(S[q.STACK_ROW_RT2NRT]).size > 2


def test_gait_stack_vs_oracle_chain_with_feedback(mpc, oracle):
    """Two robots, 300 fast ticks, against OracleNlpNode -> OracleRtNode on the CPU with the foot feedback the previous fast tick
    forwarded: /MPC/Gait to 1e-9, /rtMPC/traj to 1e-8 (relative to max(1, |value|))."""
    import torch
    nh, R, T = 10, 2, 300
    sensor, _, _ = scripted_inputs(T, R, 17)
    sensor[:, 0] = 1.0
    st = Stack(mpc, nh, R, SERVO_SLOTS)
    gaits = torch.zeros(T, 100, R, dtype=torch.float64, device="cuda"); trajs = torch.zeros_like(gaits)
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        for k in range(T):
            st.tick(planner_ticks(k), sensor[k])
            gaits[k].copy_(st.block(q.STACK_ROW_GAIT, 100)); trajs[k].copy_(st.block(q.STACK_ROW_TRAJ, 100))
    mpc.synchronize(); torch.cuda.synchronize()
    g_dev, t_dev = gaits.cpu().numpy(), trajs.cpu().numpy()
    rel = lambda a, b: np.abs(a - b) / np.maximum(1.0, np.abs(b))
    for r in range(R):
        pn, rn = OracleNlpNode(oracle), OracleRtNode(oracle, nh)
        msg, w, fb = np.zeros(100), 0, np.zeros(6)                     # fb: L xyz, R xyz of the previous fast tick
        for k in range(T):
            if planner_ticks(k):
                w += 1
                msg = pn.tick(w, 1, fb[3:6].copy(), fb[0:3].copy())
            assert rel(g_dev[k, :, r], msg).max() < 1e-9, f"robot {r} tick {k}: /MPC/Gait"
            bs = np.ascontiguousarray(sensor[k, 1:5, r])
            out = rn.tick(msg, ctrl=1, bs=bs)
            np.testing.assert_array_equal(t_dev[k, [27, 63, 98, 99], r], out[[27, 63, 98, 99]])
            assert rel(t_dev[k, :, r], out).max() < 1e-8, f"robot {r} tick {k}: /rtMPC/traj"
            fb = sensor[k, 5:11, r]
    assert (np.abs(t_dev[:, 72:86]).sum(axis=1) > 0).sum() > 100


def test_gait_stack_batch_size_changes(mpc):
    """4000 -> 1500 -> 4000 robots on one stream: the 1500-robot batch equals the first 1500 robots of the 4000-robot batch given
    the same inputs (no stale control-message rows or workspace of the larger batch)."""
    import torch
    nh, T = 10, 12
    s = torch.cuda.Stream()
    sensor, _, _ = scripted_inputs(T, 4000, 23)
    big = Stack(mpc, nh, 4000, SERVO_SLOTS, s.cuda_stream)
    small = Stack(mpc, nh, 1500, SERVO_SLOTS, s.cuda_stream)
    torch.cuda.synchronize()
    for k in range(T):
        pl = planner_ticks(k)
        big.tick(pl, sensor[k]); rb = big.rows.copy()
        small.tick(pl, np.ascontiguousarray(sensor[k][:, :1500])); rs = small.rows.copy()
        s.synchronize()
        np.testing.assert_array_equal(rs, rb[:1500])
    torch.cuda.synchronize()
    np.testing.assert_array_equal(small.state.cpu().numpy(), big.state.cpu().numpy()[:, :1500])
    np.testing.assert_array_equal(small.body_out.cpu().numpy(), big.body_out.cpu().numpy()[:1500])


def test_gait_stack_graph_capture(mpc):
    """A 5-call schedule (planner calls included) captured after warm-up replays bit-identically to the enqueued calls."""
    import torch
    nh, B, W, K = 10, 700, 8, 5
    s = torch.cuda.Stream()
    sensor, _, _ = scripted_inputs(W + K, B, 29)
    pinned = [torch.from_numpy(sensor[k].copy()).pin_memory() for k in range(W + K)]
    rows_h = [torch.zeros(B, len(SERVO_SLOTS), dtype=torch.float64).pin_memory() for _ in range(K)]
    st = Stack(mpc, nh, B, SERVO_SLOTS, s.cuda_stream)
    torch.cuda.synchronize()

    def call(k, rows):
        t = mpc.gait_stack_tick_struct(nh, planner_ticks(k), pinned[k], st.state, st.body_out, SERVO_SLOTS, st.rows_d, rows)
        mpc.gait_stack_tick_host_async(B, t, s.cuda_stream)

    for k in range(W):
        call(k, None)
    s.synchronize()
    state0, bo0 = st.state.clone(), st.body_out.clone()
    for j in range(K):
        call(W + j, rows_h[j])
    s.synchronize()
    want = [r.numpy().copy() for r in rows_h]
    want_state, want_bo = st.state.cpu().numpy(), st.body_out.cpu().numpy()
    st.state.copy_(state0); st.body_out.copy_(bo0)
    for r in rows_h:
        r.zero_()
    torch.cuda.synchronize()
    launches = mpc.launch_count
    mpc._check(mpc.lib.go1mpc_graph_capture_begin(mpc.h, s.cuda_stream), "capture_begin")
    for j in range(K):
        call(W + j, rows_h[j])
    ge = ctypes.c_void_p()
    mpc._check(mpc.lib.go1mpc_graph_capture_end(mpc.h, s.cuda_stream, ctypes.byref(ge)), "capture_end")
    assert mpc.launch_count > launches
    mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, s.cuda_stream), "graph_launch")
    s.synchronize()
    mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
    for j in range(K):
        np.testing.assert_array_equal(rows_h[j].numpy(), want[j])
    np.testing.assert_array_equal(st.state.cpu().numpy(), want_state)
    np.testing.assert_array_equal(st.body_out.cpu().numpy(), want_bo)


def test_gait_stack_rejects_bad_arguments(mpc):
    """Each bad argument returns its code and launches nothing."""
    import torch
    nh, B = 10, 64
    st = Stack(mpc, nh, B, SERVO_SLOTS)
    sensor = np.zeros((q.STACK_SENSOR_ROWS, B)); sensor[0] = 1.0
    raw = torch.zeros(B * q.body_out_stride(nh) + 2, dtype=torch.float64, device="cuda")
    ok = dict(nh=nh, planner=1, sensor=sensor, state_d=st.state, body_out_d=st.body_out, slots=SERVO_SLOTS, rows_d=st.rows_d)

    def rc(**kw):
        a = dict(ok); a.update(kw)
        t = mpc.gait_stack_tick_struct(**a)
        return mpc.lib.go1mpc_gait_stack_tick_host_async(mpc.h, B, ctypes.byref(t), None)

    cases = [
        (dict(nh=2), -4), (dict(nh=41), -4),
        (dict(slots=[]), -1), (dict(slots=[0] * 65), -1), (dict(slots=[0, 200]), -1), (dict(slots=[-1]), -1),
        (dict(sensor=None), -1), (dict(state_d=None), -1), (dict(body_out_d=None), -1), (dict(rows_d=None), -1),
        (dict(body_out_d=raw[1:].data_ptr()), -1), (dict(rows_d=st.rows_d.data_ptr() + 4), -1),
    ]
    torch.cuda.synchronize()
    before = mpc.launch_count
    for kw, code in cases:
        assert rc(**kw) == code, kw
    assert mpc.lib.go1mpc_gait_stack_tick_host_async(mpc.h, -1, None, None) == -1
    assert mpc.launch_count == before
    # the planner node needs CoM_height_solve on the device: a handle configured for external heights is refused
    h2 = q.Go1Mpc(0, cfg={"step": {"ext_height": 1}})
    try:
        t = h2.gait_stack_tick_struct(**ok)
        b2 = h2.launch_count
        assert h2.lib.go1mpc_gait_stack_tick_host_async(h2.h, B, ctypes.byref(t), None) == -4
        assert h2.launch_count == b2
    finally:
        h2.close()
    # and a valid call still works after the refusals
    rc()
    mpc.synchronize()
    assert mpc.launch_count > before
