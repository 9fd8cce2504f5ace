"""The servo stack tick (go1mpc_servo_stack_tick_async): K consecutive 1 kHz ticks of go1_servo's loop -- 9 butterworthLPF
objects on /MPC/Gait slots 0-2, 6-8, 9-11, the gait_mode leg mapping and 4 x Inverse_kinematics_g -- read in place from the
messages the gait stack keeps resident, joint targets out.

- bit for bit K x (go1mpc_lpf_batch + go1mpc_servo_kin_tick_batch) chained by hand, every gait mode, y_offset != 1;
- K splits: one K = 10 call = ten K = 1 calls = K = 3 + 7;
- the CPU oracle chain butterworthLPF -> leg mapping -> Inverse_kinematics_g;
- physics: FK of the returned joint angles puts the converged feet on their targets;
- the host interface: host copy, batch-size changes on one stream, graph capture, argument checks that launch nothing."""
import ctypes

import numpy as np
import pytest

import quadrupedal_loco_b200 as q
from tests.oracle_lib import P
from tests.test_filters import oracle_lpf
from tests.test_gpu_gait_stack import SERVO_SLOTS, Stack, planner_ticks, scripted_inputs

pytestmark = pytest.mark.gpu

NH = 10
HW = 0.12675                              # cfg.step.half_hip_width
HCOM = 0.309458                           # cfg.step.hcom
QH = np.array([0, 0.87, -1.5])            # homing pose, servo.cpp:767
RIGHT = {101: [1, 0, 1, 0], 102: [1, 0, 0, 1], 103: [1, 1, 0, 0]}   # FR, FL, RR, RL follow the right virtual foot?
WARM = 100                                # fast ticks walked before the servo starts: the body MPC's angles are live by then


def homing_feet(oracle):
    """World foot positions [12] of the homing pose with the body at the planner's CoM height (FR, FL, RR, RL xyz)."""
    hom, _ = oracle.leg_fk(np.tile(QH, (4, 1)), np.arange(4), np.tile([0, 0, HCOM], (4, 1)), np.zeros((4, 3)))
    return hom.reshape(12)


def servo_state0(oracle, B, seed):
    """Initial servo state [69][B]: the homing pose with a per-robot jitter as q, the homing feet, zero filters."""
    rng = np.random.Generator(np.random.Philox(seed))
    s = np.zeros((q.SERVO_STATE_ROWS, B))
    s[q.SERVO_ROW_Q:q.SERVO_ROW_Q + 12] = np.tile(QH, 4)[:, None] + rng.uniform(-0.05, 0.05, (12, B))
    s[q.SERVO_ROW_HOMING:q.SERVO_ROW_HOMING + 12] = homing_feet(oracle)[:, None]
    return s


def walking_inputs(T, R, seed):
    """Sensor rows [T][11][R] of scripted_inputs, robots out of phase: robot r idles for its first 5 (r % 10) fast ticks."""
    sensor, _, _ = scripted_inputs(T, R, seed)
    sensor[:, 0] = 1.0
    start = np.ones((T, R), np.int32)
    for r in range(min(R, 10)):
        start[:5 * r, r::10] = 0
    return sensor, start


def prime_filters(state, gait):
    """A servo started on a walking robot: every filter object holds the current message value (y_p, y_pp, x_p, x_pp; the call
    counter stays 0), so the filtered pose starts on the message instead of rising from zero."""
    for r5 in range(1, 5):
        state[q.SERVO_ROW_LPF + 9 * r5:q.SERVO_ROW_LPF + 9 * r5 + 9] = gait[q.SERVO_LPF_SLOTS]


def oracle_lpf_from(oracle, s0, x):
    """butterworthLPF (oracle/filters.c) on the samples x from the object state s0 = (counter, y_p, y_pp, x_p, x_pp)."""
    _, c = oracle_lpf(oracle, 1000.0, 3.0, [])
    st = np.array(s0, dtype=np.float64)
    return np.array([oracle.lib.orc_lpf_filter(ctypes.byref(c), P(st), float(v)) for v in x])


def walk(st, sensor, start, k0, k1):
    for k in range(k0, k1):
        st.tick(planner_ticks(k), sensor[k], start=np.ascontiguousarray(start[k]))


def bits(t):
    import torch
    return t.contiguous().view(torch.int64)


def test_servo_stack_equals_chained_entries(mpc, oracle):
    """4096 robots out of phase: after each of 60 fast ticks, a K = 10 call against 10 x (lpf_batch on the state's /MPC/Gait block
    with in_rows = the 9 slots, servo_kin_tick with theta = traj 72 / 73 / 0): every tick's q, the last tick's jac / foot_des /
    iters and the final servo state, bit for bit -- gait modes 101, 102, 103, y_offset 0.85, 1, 1.15; the first run's filters
    start from zero (their start-up branch), the others primed on the message."""
    import torch
    B, T, K = 4096, 60, 10
    dev = torch.device("cuda", 0)
    sensor, start = walking_inputs(WARM + T, B, 31)
    st = Stack(mpc, NH, B, SERVO_SLOTS)
    coef = np.tile(q.lpf_coefficients(1000.0, 3.0), (9, 1))
    rows9 = torch.tensor(q.SERVO_LPF_SLOTS, dtype=torch.int32, device=dev)
    zero = torch.zeros(B, dtype=torch.float64, device=dev)
    runs = []
    for i, (gm, yo) in enumerate(((101, 0.85), (102, 1.0), (103, 1.15))):
        s0 = torch.from_numpy(servo_state0(oracle, B, 40 + i)).to(dev)
        f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)
        i32 = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)
        runs.append(dict(gm=gm, yo=yo, state=s0.clone(), q_d=f64(B, 12 * K), jac=f64(36, B), fd=f64(12, B), it=i32(4, B),
                         cq=s0[0:12].clone(), hom=s0[12:24].clone(), lpf=f64(5, 9, B), out=f64(9, B),
                         cjac=f64(36, B), cfd=f64(12, B), cit=i32(4, B)))
    bad = torch.zeros((), dtype=torch.int64, device=dev)
    gait, traj = st.block(q.STACK_ROW_GAIT, 100), st.block(q.STACK_ROW_TRAJ, 100)
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        walk(st, sensor, start, 0, WARM)
        for k in range(WARM, WARM + T):
            walk(st, sensor, start, k, k + 1)
            if k == WARM:
                for r in runs[1:]:
                    prime_filters(r["state"], gait)
                    r["lpf"].copy_(r["state"][24:69].view(5, 9, B))
            theta = torch.stack([traj[72], traj[73], zero])
            for r in runs:
                mpc.servo_stack_tick(B, K, r["gm"], r["yo"], st.state, r["state"], r["q_d"], jac_d=r["jac"], foot_des_d=r["fd"],
                                     iters_d=r["it"])
                qk = r["q_d"].view(B, K, 12)
                for j in range(K):
                    mpc.lpf_batch(B, 9, coef, gait, r["lpf"], r["out"], in_rows_d=rows9)
                    o = r["out"]
                    mpc.servo_kin_tick(B, r["gm"], r["yo"], o[0:3], theta, o[6:9], o[3:6], r["hom"], r["cq"], r["cjac"], r["cfd"], r["cit"])
                    bad += (bits(qk[:, j].T) != bits(r["cq"])).sum()
    mpc.synchronize(); torch.cuda.synchronize()
    assert bad.item() == 0
    for r in runs:
        S = r["state"].cpu().numpy()
        np.testing.assert_array_equal(S[0:12], r["cq"].cpu().numpy())
        np.testing.assert_array_equal(S[12:24], r["hom"].cpu().numpy())
        np.testing.assert_array_equal(S[24:69].reshape(5, 9, B), r["lpf"].cpu().numpy())
        for a, b in (("jac", "cjac"), ("fd", "cfd"), ("it", "cit")):
            np.testing.assert_array_equal(r[a].cpu().numpy(), r[b].cpu().numpy())
        assert (r["it"].cpu().numpy() > 0).any()
        if r is not runs[0]:
            assert np.isfinite(S).all()
    # the wiring was live: walking robots, body-MPC angles non-zero, the filters past their start-up
    th = traj[72:74].cpu().numpy()
    assert (np.abs(th).sum(axis=0) > 0).mean() > 0.5
    assert (runs[0]["state"][24].cpu().numpy() == 3.0).all()


def test_servo_stack_k_split(mpc, oracle):
    """One K = 10 call = ten K = 1 calls = K = 3 + 7 calls, joint targets and final state bit for bit, over 8 fast ticks."""
    import torch
    B, T = 1000, 8
    dev = torch.device("cuda", 0)
    sensor, start = walking_inputs(WARM + T, B, 37)
    st = Stack(mpc, NH, B, SERVO_SLOTS)
    s0 = torch.from_numpy(servo_state0(oracle, B, 3)).to(dev)
    splits = ([10], [1] * 10, [3, 7])
    states = [s0.clone() for _ in splits]
    qs = [[] for _ in splits]
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        walk(st, sensor, start, 0, WARM)
        for k in range(WARM, WARM + T):
            walk(st, sensor, start, k, k + 1)
            if k == WARM:
                for sv in states:
                    prime_filters(sv, st.block(q.STACK_ROW_GAIT, 100))
            for i, ks in enumerate(splits):
                parts = []
                for K in ks:
                    qd = torch.zeros(B, 12 * K, dtype=torch.float64, device=dev)
                    mpc.servo_stack_tick(B, K, 102, 0.9, st.state, states[i], qd)
                    parts.append(qd)
                qs[i].append(torch.cat(parts, dim=1))
    mpc.synchronize(); torch.cuda.synchronize()
    want = torch.stack(qs[0]).cpu().numpy()
    for i in (1, 2):
        np.testing.assert_array_equal(torch.stack(qs[i]).cpu().numpy(), want)
        np.testing.assert_array_equal(states[i].cpu().numpy(), states[0].cpu().numpy())
    assert np.abs(np.diff(want.reshape(T, B, 10, 12), axis=2)).max() > 0      # q moves within a call


def test_servo_stack_vs_oracle_chain(mpc, oracle):
    """Sampled robots against the oracle: butterworthLPF (oracle/filters.c, from the primed state) on the held message slots, the
    numpy leg mapping and oracle.leg_ik from the previous tick's joint angles -- filtered values bit-exact, q and J to 1e-9,
    Newton counts exact."""
    import torch
    B, T, K, gm, yo = 64, 30, 10, 102, 0.85
    dev = torch.device("cuda", 0)
    sensor, start = walking_inputs(WARM + T, B, 41)
    st = Stack(mpc, NH, B, SERVO_SLOTS)
    s0 = servo_state0(oracle, B, 5)
    state = torch.from_numpy(s0.copy()).to(dev)
    q_d = torch.zeros(B, 12 * K, dtype=torch.float64, device=dev)
    jac = torch.zeros(36, B, dtype=torch.float64, device=dev); fd = torch.zeros(12, B, dtype=torch.float64, device=dev)
    it = torch.zeros(4, B, dtype=torch.int32, device=dev)
    msgs, ths, qq, ss, jj, ff, ii = [], [], [], [], [], [], []
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        walk(st, sensor, start, 0, WARM)
        for k in range(WARM, WARM + T):
            walk(st, sensor, start, k, k + 1)
            if k == WARM:
                prime_filters(state, st.block(q.STACK_ROW_GAIT, 100))
            mpc.servo_stack_tick(B, K, gm, yo, st.state, state, q_d, jac_d=jac, foot_des_d=fd, iters_d=it)
            msgs.append(st.block(q.STACK_ROW_GAIT, 100)[q.SERVO_LPF_SLOTS].clone())
            ths.append(st.block(q.STACK_ROW_TRAJ, 100)[72:74].clone())
            for lst, t in ((qq, q_d), (ss, state), (jj, jac), (ff, fd), (ii, it)):
                lst.append(t.clone())
    mpc.synchronize(); torch.cuda.synchronize()
    msgs, ths, qq, ss, jj, ff, ii = (torch.stack(v).cpu().numpy() for v in (msgs, ths, qq, ss, jj, ff, ii))
    hom = s0[12:24, 0]
    for r in (0, 13, 37, B - 1):
        filt = np.stack([oracle_lpf_from(oracle, [0.0] + [msgs[0, c, r]] * 4, np.repeat(msgs[:, c, r], K)) for c in range(9)],
                        axis=1)                                                       # [T K][9]
        np.testing.assert_array_equal(ss[:, 24 + 27:24 + 36, r], filt[K - 1::K])      # x_p after each call = its last tick's output
        qprev = s0[0:12, r]
        for k in range(T):
            for j in range(K):
                f = filt[k * K + j]
                bp = np.array([[f[0], f[1] * yo, f[2]]]); br = np.array([[ths[k, 0, r], ths[k, 1, r], 0.0]])
                qg = qq[k, r, 12 * j:12 * j + 12]
                for leg in range(4):
                    right = RIGHT[gm][leg]
                    pdes = hom[3 * leg:3 * leg + 3] + (f[6:9] if right else f[3:6])
                    pdes[1] += HW if right else -HW
                    qo, Jo, ito = oracle.leg_ik(pdes[None], qprev[None, 3 * leg:3 * leg + 3], [leg], bp, br)
                    np.testing.assert_allclose(qg[3 * leg:3 * leg + 3], qo[0], rtol=0, atol=1e-9)
                    if j == K - 1:
                        np.testing.assert_array_equal(ff[k, 3 * leg:3 * leg + 3, r], pdes)
                        np.testing.assert_allclose(jj[k, 9 * leg:9 * leg + 9, r], Jo[0], rtol=0, atol=1e-9)
                        assert ii[k, leg, r] == ito[0], (r, k, leg)
                qprev = qg
    assert np.abs(ths[-1]).max() > 0
    # the filters ran from zero as well: the first robot's first call against oracle_lpf from a fresh object
    sz = torch.from_numpy(s0.copy()).to(dev)
    mpc.servo_stack_tick(B, K, gm, yo, st.state, sz, q_d)
    mpc.synchronize()
    last = st.block(q.STACK_ROW_GAIT, 100)[q.SERVO_LPF_SLOTS, 0].cpu().numpy()
    want = [oracle_lpf(oracle, 1000.0, 3.0, np.full(K, last[c]))[0][-1] for c in range(9)]
    np.testing.assert_array_equal(sz[24 + 27:24 + 36, 0].cpu().numpy(), want)


def test_servo_stack_feet_on_targets(mpc, oracle):
    """Physics: for converged legs (iters < 15) oracle FK of the returned q with the body pose of the last tick puts the feet on
    foot_des within the solver's stop radius |dp| <= 1e-3."""
    import torch
    B, T, K, gm, yo = 4096, 30, 10, 101, 0.9
    dev = torch.device("cuda", 0)
    sensor, start = walking_inputs(WARM + T, B, 43)
    st = Stack(mpc, NH, B, SERVO_SLOTS)
    state = torch.from_numpy(servo_state0(oracle, B, 7)).to(dev)
    q_d = torch.zeros(B, 12 * K, dtype=torch.float64, device=dev)
    fd = torch.zeros(12, B, dtype=torch.float64, device=dev); it = torch.zeros(4, B, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        walk(st, sensor, start, 0, WARM)
        for k in range(WARM, WARM + T):
            walk(st, sensor, start, k, k + 1)
            if k == WARM:
                prime_filters(state, st.block(q.STACK_ROW_GAIT, 100))
            mpc.servo_stack_tick(B, K, gm, yo, st.state, state, q_d, foot_des_d=fd, iters_d=it)
    mpc.synchronize(); torch.cuda.synchronize()
    S, fd, it = state.cpu().numpy(), fd.cpu().numpy(), it.cpu().numpy()
    traj = st.block(q.STACK_ROW_TRAJ, 100).cpu().numpy()
    com = S[24 + 27:24 + 30]                                     # x_p of channels 0..2: the last tick's filtered CoM
    n = 400
    bp = np.stack([com[0], com[1] * yo, com[2]], axis=1)[:n]
    br = np.stack([traj[72], traj[73], np.zeros(B)], axis=1)[:n]
    conv = it[:, :n] < 15
    for leg in range(4):
        pos, _ = oracle.leg_fk(S[3 * leg:3 * leg + 3, :n].T, np.full(n, leg), bp, br)
        err = np.linalg.norm(pos - fd[3 * leg:3 * leg + 3, :n].T, axis=1)
        assert err[conv[leg]].max() <= 1.0000001e-3, leg
    assert conv.mean() > 0.5, conv.mean()
    np.testing.assert_array_equal(S[0:12], q_d.cpu().numpy()[:, -12:].T)


def test_servo_stack_host_copy_and_batch_size_changes(mpc, oracle):
    """The host copy equals q_d; 4000 -> 1500 -> 4000 robots on one stream: the 1500-robot batch equals the first 1500 robots of
    the 4000-robot batch given the same inputs."""
    import torch
    T, K = 6, 10
    s = torch.cuda.Stream()
    sensor, start = walking_inputs(WARM + T, 4000, 47)
    big, small = Stack(mpc, NH, 4000, SERVO_SLOTS, s.cuda_stream), Stack(mpc, NH, 1500, SERVO_SLOTS, s.cuda_stream)
    s0 = servo_state0(oracle, 4000, 9)
    sb = torch.from_numpy(s0.copy()).cuda(); ss = torch.from_numpy(np.ascontiguousarray(s0[:, :1500])).cuda()
    qb = torch.zeros(4000, 12 * K, dtype=torch.float64, device="cuda"); qs = torch.zeros(1500, 12 * K, dtype=torch.float64, device="cuda")
    hb = torch.zeros(4000, 12 * K, dtype=torch.float64).pin_memory(); hs = torch.zeros(1500, 12 * K, dtype=torch.float64).pin_memory()
    torch.cuda.synchronize()
    for k in range(WARM + T):
        pl = planner_ticks(k)
        big.tick(pl, sensor[k], start=np.ascontiguousarray(start[k]))
        small.tick(pl, np.ascontiguousarray(sensor[k][:, :1500]), start=np.ascontiguousarray(start[k][:1500]))
        if k >= WARM:
            mpc.servo_stack_tick(4000, K, 103, 1.0, big.state, sb, qb, q=hb, stream=s.cuda_stream)
            mpc.servo_stack_tick(1500, K, 103, 1.0, small.state, ss, qs, q=hs, stream=s.cuda_stream)
            s.synchronize()
            np.testing.assert_array_equal(hb.numpy(), qb.cpu().numpy())
            np.testing.assert_array_equal(hs.numpy(), qs.cpu().numpy())
            np.testing.assert_array_equal(hs.numpy(), hb.numpy()[:1500])
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ss.cpu().numpy(), sb.cpu().numpy()[:, :1500])


def test_servo_stack_graph_capture(mpc, oracle):
    """A warmed-up 10 ms period -- gait stack tick, then the K = 10 servo call with the joint targets down -- captured for 4
    periods replays bit-identically to the enqueued calls."""
    import torch
    B, W, P, K = 700, WARM, 4, 10
    s = torch.cuda.Stream()
    sensor, start = walking_inputs(W + P, B, 53)
    pinned = [torch.from_numpy(sensor[k].copy()).pin_memory() for k in range(W + P)]
    q_h = [torch.zeros(B, 12 * K, dtype=torch.float64).pin_memory() for _ in range(P)]
    st = Stack(mpc, NH, B, SERVO_SLOTS, s.cuda_stream)
    sv = torch.from_numpy(servo_state0(oracle, B, 11)).cuda()
    q_d = torch.zeros(B, 12 * K, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()

    def period(k, qh):
        t = mpc.gait_stack_tick_struct(NH, planner_ticks(k), pinned[k], st.state, st.body_out, SERVO_SLOTS, st.rows_d, None)
        mpc.gait_stack_tick_host_async(B, t, s.cuda_stream)
        if qh is not None:
            mpc.servo_stack_tick(B, K, 102, 0.95, st.state, sv, q_d, q=qh, stream=s.cuda_stream)

    for k in range(W):
        period(k, None if k < W - 5 else q_h[0])
    s.synchronize()
    snap = [t.clone() for t in (st.state, st.body_out, sv)]
    for j in range(P):
        period(W + j, q_h[j])
    s.synchronize()
    want = [h.numpy().copy() for h in q_h]
    want_state = [t.cpu().numpy() for t in (st.state, st.body_out, sv)]
    for t, c in zip((st.state, st.body_out, sv), snap):
        t.copy_(c)
    for h in q_h:
        h.zero_()
    torch.cuda.synchronize()
    mpc._check(mpc.lib.go1mpc_graph_capture_begin(mpc.h, s.cuda_stream), "capture_begin")
    for j in range(P):
        period(W + j, q_h[j])
    ge = ctypes.c_void_p()
    mpc._check(mpc.lib.go1mpc_graph_capture_end(mpc.h, s.cuda_stream, ctypes.byref(ge)), "capture_end")
    mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, s.cuda_stream), "graph_launch")
    s.synchronize()
    mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
    for j in range(P):
        np.testing.assert_array_equal(q_h[j].numpy(), want[j])
    for t, w in zip((st.state, st.body_out, sv), want_state):
        np.testing.assert_array_equal(t.cpu().numpy(), w)


def test_servo_stack_rejects_bad_arguments(mpc, oracle):
    """Each bad argument returns its code, launches nothing and leaves q_d and the servo state untouched."""
    import torch
    B, K = 64, 10
    st = Stack(mpc, NH, B, SERVO_SLOTS)
    sv = torch.from_numpy(servo_state0(oracle, B, 13)).cuda()
    raw = torch.full((B * 12 * K + 1,), 7.0, dtype=torch.float64, device="cuda")
    q_d = raw[:-1].view(B, 12 * K)
    ok = dict(K=K, gait_mode=102, y_offset=1.0, stack_state_d=st.state, servo_state_d=sv, q_d=q_d)

    def rc(B=B, **kw):
        a = dict(ok); a.update(kw)
        t = mpc.servo_stack_tick_struct(**a)
        return mpc.lib.go1mpc_servo_stack_tick_async(mpc.h, B, ctypes.byref(t), None)

    cases = [
        (dict(K=0), -1), (dict(K=11), -1), (dict(K=-3), -1),
        (dict(stack_state_d=None), -1), (dict(servo_state_d=None), -1), (dict(q_d=None), -1),
        (dict(q_d=raw.data_ptr() + 4), -1),
        (dict(gait_mode=100), -4), (dict(gait_mode=104), -4), (dict(gait_mode=0), -4),
    ]
    torch.cuda.synchronize()
    sv0, q0 = sv.cpu().numpy(), q_d.cpu().numpy()
    before = mpc.launch_count
    for kw, code in cases:
        assert rc(**kw) == code, kw
    assert rc(B=-1) == -1
    assert mpc.lib.go1mpc_servo_stack_tick_async(mpc.h, 5, None, None) == -1
    assert mpc.lib.go1mpc_servo_stack_tick_async(mpc.h, 0, None, None) == 0      # B = 0: no-op
    assert rc(B=0) == 0
    mpc.synchronize(); torch.cuda.synchronize()
    assert mpc.launch_count == before
    np.testing.assert_array_equal(sv.cpu().numpy(), sv0)
    np.testing.assert_array_equal(q_d.cpu().numpy(), q0)
    # and a valid call still works after the refusals
    assert rc() == 0
    mpc.synchronize()
    assert mpc.launch_count == before + 1
    assert not (q_d.cpu().numpy() == 7.0).any()
