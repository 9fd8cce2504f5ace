"""The servo torque tick (go1mpc_servo_torque_tick_async): the servo stack's K ticks, each followed by force_distribution, the
12-variable force QP and the four-leg torque map, with the force state resident on the device.

- joint targets and servo state bit-identical to go1mpc_servo_stack_tick_async, gait modes 101, 102, 103;
- tick by tick bit for bit against the chained single-stage entries (K = 1 servo stack, leg FK, force distribution, force QP,
  joint torques) wired as the header documents, at B = 1, 257, 3000;
- K splits with the force state carried; the CPU oracle chain; QP invariants; resets; one captured period graph; batch-size
  changes and argument refusal."""
import ctypes

import numpy as np
import pytest

import quadrupedal_loco_b200 as q
from tests.test_gpu_gait_stack import SERVO_SLOTS, Stack, planner_ticks
from tests.test_gpu_gait_stack_clocked import Farm, servo_columns
from tests.test_gpu_servo_stack import QH, prime_filters, servo_state0, walk, walking_inputs

pytestmark = pytest.mark.gpu

NH = 10
WARM = 100
YC = 0.9                                      # force_distribution's y_coefficient
RIGHT = {101: [1, 0, 1, 0], 102: [1, 0, 0, 1], 103: [1, 1, 0, 0]}
LPF_XP = q.SERVO_ROW_LPF + 27                 # row of channel 0's x_p (the filter's last output) in the servo state


def bits(t):
    import torch
    return t.contiguous().view(torch.int64)


def meas0(B, seed):
    """Measured joints [24][B]: the homing pose with a per-robot jitter, joint velocities of a few rad/s."""
    rng = np.random.Generator(np.random.Philox(seed))
    m = np.zeros((24, B))
    m[:12] = np.tile(QH, 4)[:, None] + rng.uniform(-0.1, 0.1, (12, B))
    m[12:] = rng.uniform(-3.0, 3.0, (12, B))
    return m


def swing_legs(gm, rs):
    """[4][B] int32: the QP's zero-force rule per leg (FR, FL, RR, RL)."""
    rs = rs.astype(np.int64)
    if gm == 102:
        mask = np.where(rs == 0, 0x6, np.where(rs == 1, 0x9, 0))
    elif gm == 101:
        mask = np.where(rs == 0, 0x5, np.where(rs == 1, 0xA, 0))
    else:
        mask = np.zeros_like(rs)
    return np.stack([(mask >> l) & 1 for l in range(4)]).astype(np.int32)


class Torque:
    """One batch's torque-tick buffers: servo state, force state, measurements, outputs."""

    def __init__(self, B, K, servo, meas):
        import torch
        dev = torch.device("cuda", 0)
        f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)
        self.B, self.K = B, K
        self.servo = torch.from_numpy(np.ascontiguousarray(servo)).to(dev)
        self.force = f64(q.SERVO_FORCE_ROWS, B)
        self.meas = torch.from_numpy(np.ascontiguousarray(meas)).to(dev)
        self.q_d, self.tau_d = f64(B, 12 * K), f64(B, 12 * K)
        self.grf, self.diag = f64(B, 16), torch.zeros(B, 32, dtype=torch.int32, device=dev)

    def call(self, mpc, state, gm, yo, K=None, q_d=None, tau_d=None, stream=None, **kw):
        mpc.servo_torque_tick(self.B, K or self.K, gm, yo, YC, state, self.servo, self.force, self.meas,
                              self.q_d if q_d is None else q_d, self.tau_d if tau_d is None else tau_d, stream=stream, grf_d=self.grf,
                              grf_diag_d=self.diag, **kw)


class Chain:
    """The same ticks from the single-stage entries: K = 1 servo stack calls, leg FK, force distribution / QP / torque map."""

    def __init__(self, mpc, B, servo, meas):
        import torch
        dev = torch.device("cuda", 0)
        f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)
        self.mpc, self.B = mpc, B
        self.servo = torch.from_numpy(np.ascontiguousarray(servo)).to(dev)
        self.meas = torch.from_numpy(np.ascontiguousarray(meas)).to(dev)
        self.q1, self.jac, self.fd = f64(B, 12), f64(36, B), f64(12, B)
        self.fref, self.prev = f64(12, B), f64(B, 12)
        self.rec, self.out, self.diag = f64(B, 48), f64(B, 16), torch.zeros(B, 32, dtype=torch.int32, device=dev)
        self.tau, self.pos, self.mjac = f64(12, B), f64(3, 4 * B), f64(9, 4 * B)
        self.legs = torch.arange(4, dtype=torch.int32, device=dev).repeat_interleave(B)
        self.qm = self.meas[:12].view(4, 3, B).permute(1, 0, 2).reshape(3, 4 * B).contiguous()
        self.dq = self.meas[12:].view(4, 3, B)

    def tick(self, state, gm, yo):
        """One 1 kHz tick; returns q [B][12] and tau [12][B] (views of the chain's buffers)."""
        import torch
        mpc, B = self.mpc, self.B
        mpc.servo_stack_tick(B, 1, gm, yo, state, self.servo, self.q1, jac_d=self.jac, foot_des_d=self.fd)
        ch = self.servo[LPF_XP:LPF_XP + 9]
        gait = state[q.STACK_ROW_GAIT:q.STACK_ROW_GAIT + 100]
        traj = state[q.STACK_ROW_TRAJ:q.STACK_ROW_TRAJ + 100]
        com = torch.stack([ch[0], ch[1] * yo, ch[2]])
        if gm in (101, 102):
            mpc.grf_force_distribution(B, gm, YC, com, self.fd, gait[15:21].contiguous(), ch[6:9].contiguous(), ch[3:6].contiguous(),
                                       self.fref)
        r = self.rec
        r.zero_()
        r[:, 0:3] = com.T; r[:, 3:15] = self.fd.T
        r[:, 15:18] = (gait[15:18] + gait[18:21]).T; r[:, 18:21] = (gait[21:24] + gait[24:27]).T
        r[:, 21:33] = self.fref.T; r[:, 33:45] = self.prev; r[:, 45] = gm; r[:, 46] = gait[99]
        mpc.grf_force_opt(B, r, self.out, self.diag)
        bp = com.repeat(1, 4).contiguous()
        br = torch.stack([traj[72], traj[73], torch.zeros_like(traj[72])]).repeat(1, 4).contiguous()
        mpc.leg_fk(4 * B, self.qm, self.legs, bp, br, self.pos, self.mjac)
        J = self.mjac.view(9, 4, B)
        pest = self.pos.view(3, 4, B).permute(1, 0, 2).reshape(12, B).contiguous()
        pvest = torch.stack([(J[3 * i] * self.dq[:, 0] + J[3 * i + 1] * self.dq[:, 1]) + J[3 * i + 2] * self.dq[:, 2]
                             for i in range(3)], dim=1).reshape(12, B).contiguous()
        pvdes = torch.cat([gait[46:49] if RIGHT[gm][l] else gait[49:52] for l in range(4)]).contiguous()
        swing = torch.from_numpy(swing_legs(gm, gait[99].cpu().numpy())).to(self.out.device)
        mpc.grf_joint_torques(B, self.jac, swing, self.fd, pest, pvdes, pvest, self.out, self.tau, F_strides=(1, 16))
        self.prev.copy_(self.out[:, :12])
        return self.q1, self.tau


def set_right_support(gait, k):
    """/MPC/Gait 99 (right_support) = 0, 1, 2 across the robots, shifted by k; returns the old row.  The walked gait holds every
    robot in one support phase at a time, so the wiring of all three values is tested on one message; the 100 Hz node reads
    slot 99, so the caller restores it before the next gait stack call."""
    import torch
    old = gait[99].clone()
    gait[99] = torch.remainder(torch.arange(gait.shape[1], device=gait.device) + k, 3).to(gait.dtype)
    return old


def walked(mpc, B, seed, T):
    sensor, start = walking_inputs(WARM + T, B, seed)
    st = Stack(mpc, NH, B, SERVO_SLOTS)
    walk(st, sensor, start, 0, WARM)
    return st, sensor, start


@pytest.mark.parametrize("B", [1, 257, 3000])
def test_servo_torque_equals_chained_entries(mpc, oracle, B):
    """Every tick's q and tau, the last tick's GRF records and diagnostics, the servo and force states: bit for bit against the
    chained entries, gait modes 101 / 102 / 103, over 4 periods of K = 10 on a walked gait stack."""
    import torch
    K, T = 10, 4
    torch.cuda.synchronize()
    seen_rs, fmax = set(), 0.0
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        st, sensor, start = walked(mpc, B, 61, T)
        gait = st.block(q.STACK_ROW_GAIT, 100)
        s0 = servo_state0(oracle, B, 17)
        prime_filters(s0, gait.cpu().numpy())
        m0 = meas0(B, 19)
        runs = [(gm, 0.95, Torque(B, K, s0, m0), Chain(mpc, B, s0, m0)) for gm in (101, 102, 103)]
        bad = torch.zeros((), dtype=torch.int64, device="cuda")
        for k in range(WARM, WARM + T):
            walk(st, sensor, start, k, k + 1)
            rs_old = set_right_support(gait, k)
            seen_rs |= set(np.unique(gait[99].cpu().numpy()).tolist())
            fmax = max(fmax, float(gait[15:27].abs().max()))
            for gm, yo, tq, ch in runs:
                tq.call(mpc, st.state, gm, yo)
                for j in range(K):
                    q1, tau = ch.tick(st.state, gm, yo)
                    bad += (bits(tq.q_d[:, 12 * j:12 * j + 12]) != bits(q1)).sum()
                    bad += (bits(tq.tau_d[:, 12 * j:12 * j + 12]) != bits(tau.T)).sum()
                bad += (bits(tq.grf) != bits(ch.out)).sum() + (tq.diag != ch.diag).sum()
                bad += (bits(tq.servo) != bits(ch.servo)).sum()
                bad += (bits(tq.force[:12].T) != bits(ch.prev)).sum() + (bits(tq.force[12:]) != bits(ch.fref)).sum()
            gait[99] = rs_old
    mpc.synchronize(); torch.cuda.synchronize()
    assert bad.item() == 0
    for gm, _, tq, _ in runs:
        assert np.isfinite(tq.tau_d.cpu().numpy()).all(), gm
    if B > 1:
        assert {0.0, 1.0, 2.0} <= seen_rs, seen_rs
    assert fmax > 0


def test_servo_torque_joint_targets_unchanged(mpc, oracle):
    """q_d, jac / foot_des / iters and the servo state equal go1mpc_servo_stack_tick_async's, bit for bit."""
    import torch
    B, K, T = 2000, 10, 5
    dev = torch.device("cuda", 0)
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        st, sensor, start = walked(mpc, B, 63, T)
        s0 = servo_state0(oracle, B, 21)
        for gm in (101, 102, 103):
            tq = Torque(B, K, s0, meas0(B, 23))
            ref = torch.from_numpy(s0).to(dev)
            qd = torch.zeros(B, 12 * K, dtype=torch.float64, device=dev)
            outs = [[torch.zeros(36, B, dtype=torch.float64, device=dev), torch.zeros(12, B, dtype=torch.float64, device=dev),
                     torch.zeros(4, B, dtype=torch.int32, device=dev)] for _ in range(2)]
            st2 = Stack(mpc, NH, B, SERVO_SLOTS)
            st2.state.copy_(st.state); st2.body_out.copy_(st.body_out)
            for k in range(WARM, WARM + T):
                walk(st2, sensor, start, k, k + 1)
                tq.call(mpc, st2.state, gm, 1.05, jac_d=outs[0][0], foot_des_d=outs[0][1], iters_d=outs[0][2])
                mpc.servo_stack_tick(B, K, gm, 1.05, st2.state, ref, qd, jac_d=outs[1][0], foot_des_d=outs[1][1], iters_d=outs[1][2])
                torch.cuda.current_stream().synchronize()
                np.testing.assert_array_equal(tq.q_d.cpu().numpy(), qd.cpu().numpy())
            np.testing.assert_array_equal(tq.servo.cpu().numpy(), ref.cpu().numpy())
            for a, b in zip(*outs):
                np.testing.assert_array_equal(a.cpu().numpy(), b.cpu().numpy())


def test_servo_torque_k_split(mpc, oracle):
    """One K = 10 call = ten K = 1 calls = K = 3 + 7 calls: q, tau, servo and force states bit for bit over 5 periods."""
    import torch
    B, T, gm = 1000, 5, 102
    dev = torch.device("cuda", 0)
    torch.cuda.synchronize()
    splits = ([10], [1] * 10, [3, 7])
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        st, sensor, start = walked(mpc, B, 67, T)
        s0 = servo_state0(oracle, B, 25)
        prime_filters(s0, st.block(q.STACK_ROW_GAIT, 100).cpu().numpy())
        tqs = [Torque(B, 10, s0, meas0(B, 27)) for _ in splits]
        res = [[] for _ in splits]
        for k in range(WARM, WARM + T):
            walk(st, sensor, start, k, k + 1)
            for i, ks in enumerate(splits):
                qs, ts = [], []
                for K in ks:
                    qd = torch.zeros(B, 12 * K, dtype=torch.float64, device=dev); td = torch.zeros_like(qd)
                    tqs[i].call(mpc, st.state, gm, 0.9, K=K, q_d=qd, tau_d=td)
                    qs.append(qd); ts.append(td)
                res[i].append(torch.cat(qs + ts, dim=1))
    mpc.synchronize(); torch.cuda.synchronize()
    want = torch.stack(res[0]).cpu().numpy()
    for i in (1, 2):
        np.testing.assert_array_equal(torch.stack(res[i]).cpu().numpy(), want)
        np.testing.assert_array_equal(tqs[i].force.cpu().numpy(), tqs[0].force.cpu().numpy())
        np.testing.assert_array_equal(tqs[i].servo.cpu().numpy(), tqs[0].servo.cpu().numpy())
    assert np.abs(want[..., 120:]).max() > 0


def test_servo_torque_vs_oracle_and_invariants(mpc, oracle):
    """Sampled robots against oracle/grf.c (force_distribution + force_opt) and the oracle leg FK on the device's own tick inputs:
    1e-9 and identical active sets; where the QP converged, swing legs carry exactly 0, fz in [0, 160] and the friction pyramid
    holds to 1e-9."""
    import torch
    from tests.test_grf import oracle_grf
    B, K, gm, yo = 512, 1, 102, 1.0
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        st, sensor, start = walked(mpc, B, 71, 3)
        s0 = servo_state0(oracle, B, 29)
        prime_filters(s0, st.block(q.STACK_ROW_GAIT, 100).cpu().numpy())
        m0 = meas0(B, 31)
        tq = Torque(B, K, s0, m0)
        walk(st, sensor, start, WARM, WARM + 1)
        set_right_support(st.block(q.STACK_ROW_GAIT, 100), 0)
        prev = tq.force.clone()
        jac = torch.zeros(36, B, dtype=torch.float64, device="cuda"); fd = torch.zeros(12, B, dtype=torch.float64, device="cuda")
        tq.call(mpc, st.state, gm, yo, jac_d=jac, foot_des_d=fd)
    mpc.synchronize(); torch.cuda.synchronize()
    S, gait, traj = tq.servo.cpu().numpy(), st.block(q.STACK_ROW_GAIT, 100).cpu().numpy(), st.block(q.STACK_ROW_TRAJ, 100).cpu().numpy()
    fd, grf, dg, F = fd.cpu().numpy(), tq.grf.cpu().numpy(), tq.diag.cpu().numpy(), tq.force.cpu().numpy()
    ch = S[LPF_XP:LPF_XP + 9]
    com = np.stack([ch[0], ch[1] * yo, ch[2]], axis=1)
    d = dict(mode=np.full(B, gm), rs=gait[99].astype(np.int32), base=com, legs=fd.T.copy(),
             FT=np.concatenate([(gait[15:18] + gait[18:21]).T, (gait[21:24] + gait[24:27]).T], axis=1),
             F6=gait[15:21].T.copy(), rf=ch[6:9].T.copy(), lf=ch[3:6].T.copy(), prev=prev[:12].cpu().numpy().T.copy())
    o = oracle_grf(oracle, d, yc=YC)
    np.testing.assert_allclose(F[12:].T, o["Fg"], rtol=0, atol=1e-9)
    conv = (dg[:, 0] == 0) & (o["status"] == 0)
    assert conv.mean() > 0.9
    sc = np.maximum(1.0, np.abs(o["grf"]).max(axis=1, keepdims=True))
    assert (np.abs(grf[:, :12] - o["grf"]) / sc)[conv].max() < 1e-9
    np.testing.assert_array_equal(dg[conv, 1], o["nactive"][conv])
    for b in np.nonzero(conv)[0]:
        na = dg[b, 1]
        assert sorted(dg[b, 8:8 + na]) == sorted(o["active"][b, :na]), b
    # measured FK: the torque of a swing leg is -J' (kp (p_des - p_est) + kd (pv_des - pv_est)) + gravity term
    sw = swing_legs(gm, gait[99])
    tau = tq.tau_d.cpu().numpy()
    br = np.stack([traj[72], traj[73], np.zeros(B)], axis=1)
    Jq = jac.cpu().numpy()
    m = m0
    n_sw = 0
    for b in range(0, B, 7):
        for l in range(4):
            if not sw[l, b]:
                continue
            n_sw += 1
            pe, Jm = oracle.leg_fk(m[3 * l:3 * l + 3, b][None], [l], com[b][None], br[b][None])
            pv = Jm[0].reshape(3, 3) @ m[12 + 3 * l:15 + 3 * l, b]
            pvd = gait[46:49, b] if RIGHT[gm][l] else gait[49:52, b]
            wv = 1.0 * (fd[3 * l:3 * l + 3, b] - pe[0]) + 0.01 * (pvd - pv)
            t = -Jq[9 * l:9 * l + 9, b].reshape(3, 3).T @ wv + np.array([0.8 if l & 1 else -0.8, 0, 0])
            np.testing.assert_allclose(tau[b, 3 * l:3 * l + 3], t, rtol=0, atol=1e-9)
    assert n_sw > 0
    # invariants of the converged QPs
    x = grf[conv, :12].reshape(-1, 4, 3)
    swc = sw.T[conv].astype(bool)
    assert np.abs(x[swc]).max(initial=0.0) <= 1e-12
    fz = x[..., 2]
    assert (fz >= -1e-9).all() and (fz <= 160 + 1e-9).all()
    assert (np.abs(x[..., 0]) <= 0.25 * fz + 1e-9).all() and (np.abs(x[..., 1]) <= 0.25 * fz + 1e-9).all()


def test_servo_torque_reset(mpc, oracle):
    """Flagged robots equal a fresh zero force state; the others are bit-identical to a run without the reset."""
    import torch
    B, K, gm = 600, 10, 101
    torch.cuda.synchronize()
    flags = torch.zeros(B, dtype=torch.int32).pin_memory()
    flags[::3] = 1
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        st, sensor, start = walked(mpc, B, 73, 3)
        s0 = servo_state0(oracle, B, 33)
        m0 = meas0(B, 35)
        a, b_ = Torque(B, K, s0, m0), Torque(B, K, s0, m0)
        for k in range(WARM, WARM + 2):
            walk(st, sensor, start, k, k + 1)
            a.call(mpc, st.state, gm, 1.0); b_.call(mpc, st.state, gm, 1.0)
        walk(st, sensor, start, WARM + 2, WARM + 3)
        fresh = Torque(B, K, b_.servo.cpu().numpy(), m0)          # the same servo state, zero force state
        a.call(mpc, st.state, gm, 1.0)
        b_.call(mpc, st.state, gm, 1.0, reset=flags)
        fresh.call(mpc, st.state, gm, 1.0)
    mpc.synchronize(); torch.cuda.synchronize()
    f = flags.numpy().astype(bool)
    for t in ("tau_d", "q_d", "grf"):
        A, Bv, Fr = (getattr(x, t).cpu().numpy() for x in (a, b_, fresh))
        np.testing.assert_array_equal(Bv[f], Fr[f])
        np.testing.assert_array_equal(Bv[~f], A[~f])
    Fa, Fb, Ff = (x.force.cpu().numpy() for x in (a, b_, fresh))
    np.testing.assert_array_equal(Fb[:, f], Ff[:, f])
    np.testing.assert_array_equal(Fb[:, ~f], Fa[:, ~f])
    assert (a.tau_d.cpu().numpy()[f] != b_.tau_d.cpu().numpy()[f]).any()


def test_servo_torque_graph_capture(mpc, oracle):
    """One captured period -- gait stack reset, clocked tick, K = 10 torque tick with q and tau down -- replayed 30 times equals
    the same calls made eagerly."""
    import torch
    B, P, K = 300, 30, 10
    s = torch.cuda.Stream()
    sensor, start = walking_inputs(P + 5, B, 79)
    servo = servo_columns(oracle, B, 81, False)

    def make():
        f = Farm(mpc, B, servo, s.cuda_stream)
        return f, Torque(B, K, servo, meas0(B, 83))

    flags = torch.zeros(B, dtype=torch.int32).pin_memory()
    sens = torch.zeros(11, B, dtype=torch.float64).pin_memory()
    qh = torch.zeros(B, 12 * K, dtype=torch.float64).pin_memory(); th = torch.zeros_like(qh).pin_memory()

    def period(f, tq):
        f.reset(flags)
        f.tick(sens)
        tq.servo = f.servo
        tq.call(mpc, f.state, 102, 1.0, reset=flags, stream=s.cuda_stream, q=qh, tau=th)

    def load(k):
        sens.copy_(torch.from_numpy(np.ascontiguousarray(sensor[k])))
        flags.zero_()
        if k % 7 == 3:
            flags[k % 5::11] = 1

    runs = []
    for graph in (False, True):
        f, tq = make()
        torch.cuda.synchronize()
        load(0); period(f, tq); s.synchronize()          # warm-up: allocations, default column
        ge = None
        if graph:
            mpc._check(mpc.lib.go1mpc_graph_capture_begin(mpc.h, s.cuda_stream), "capture_begin")
            period(f, tq)
            ge = ctypes.c_void_p()
            mpc._check(mpc.lib.go1mpc_graph_capture_end(mpc.h, s.cuda_stream, ctypes.byref(ge)), "capture_end")
        hist = []
        for k in range(1, P + 1):
            load(k)
            if graph:
                mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, s.cuda_stream), "graph_launch")
            else:
                period(f, tq)
            s.synchronize()
            hist.append((qh.numpy().copy(), th.numpy().copy()))
        if graph:
            mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
        runs.append((hist, tq.force.cpu().numpy(), f.servo.cpu().numpy()))
    (h0, f0, s0), (h1, f1, s1) = runs
    for (qa, ta), (qb, tb) in zip(h0, h1):
        np.testing.assert_array_equal(qa, qb); np.testing.assert_array_equal(ta, tb)
    np.testing.assert_array_equal(f0, f1); np.testing.assert_array_equal(s0, s1)
    assert np.abs(h0[-1][1]).max() > 0


def test_servo_torque_batch_size_and_bad_arguments(mpc, oracle):
    """1500 -> 4000 robots on one stream, the small batch fed the first 1500 columns of the big one's gait stack state: its
    outputs equal the big batch's first 1500 robots.  Each bad argument returns its code, launches nothing and writes nothing."""
    import torch
    K = 10
    s = torch.cuda.Stream()
    sensor, start = walking_inputs(WARM + 2, 4000, 87)
    big = Stack(mpc, NH, 4000, SERVO_SLOTS, s.cuda_stream)
    s0, m0 = servo_state0(oracle, 4000, 89), meas0(4000, 91)
    tb, ts = Torque(4000, K, s0, m0), Torque(1500, K, s0[:, :1500], m0[:, :1500])
    torch.cuda.synchronize()
    for k in range(WARM + 2):
        big.tick(planner_ticks(k), sensor[k], start=np.ascontiguousarray(start[k]))
        if k >= WARM:
            with torch.cuda.stream(s):
                small_state = big.state[:, :1500].contiguous()
            ts.call(mpc, small_state, 103, 1.0, stream=s.cuda_stream)
            tb.call(mpc, big.state, 103, 1.0, stream=s.cuda_stream)
    s.synchronize()
    for t in ("tau_d", "q_d", "grf", "diag"):
        np.testing.assert_array_equal(getattr(ts, t).cpu().numpy(), getattr(tb, t).cpu().numpy()[:1500])
    np.testing.assert_array_equal(ts.force.cpu().numpy(), tb.force.cpu().numpy()[:, :1500])

    B = 64
    st = Stack(mpc, NH, B, SERVO_SLOTS)
    tq = Torque(B, K, servo_state0(oracle, B, 93), meas0(B, 95))
    raw = torch.full((B * 12 * K + 1,), 7.0, dtype=torch.float64, device="cuda")
    tq.q_d = raw[:-1].view(B, 12 * K)
    tq.tau_d.fill_(7.0); tq.force.fill_(7.0)
    ok = dict(K=K, gait_mode=102, y_offset=1.0, y_coefficient=YC, stack_state_d=st.state, servo_state_d=tq.servo,
              force_state_d=tq.force, meas_d=tq.meas, q_d=tq.q_d, tau_d=tq.tau_d, grf_d=tq.grf)

    def rc(B=B, **kw):
        a = dict(ok); a.update(kw)
        return mpc.lib.go1mpc_servo_torque_tick_async(mpc.h, B, ctypes.byref(mpc.servo_torque_tick_struct(**a)), None)

    cases = [
        (dict(K=0), -1), (dict(K=11), -1),
        (dict(stack_state_d=None), -1), (dict(servo_state_d=None), -1), (dict(q_d=None), -1), (dict(force_state_d=None), -1),
        (dict(meas_d=None), -1), (dict(tau_d=None), -1),
        (dict(q_d=raw.data_ptr() + 4), -1), (dict(tau_d=tq.tau_d.data_ptr() + 4), -1),
        (dict(gait_mode=100), -4), (dict(gait_mode=104), -4),
    ]
    torch.cuda.synchronize()
    before = [t.cpu().numpy() for t in (tq.servo, tq.force, tq.q_d, tq.tau_d, tq.grf)]
    n0 = mpc.launch_count
    for kw, code in cases:
        assert rc(**kw) == code, kw
    assert rc(B=-1) == -1
    assert mpc.lib.go1mpc_servo_torque_tick_async(mpc.h, 5, None, None) == -1
    assert mpc.lib.go1mpc_servo_torque_tick_async(mpc.h, 0, None, None) == 0
    assert rc(B=0) == 0
    mpc.synchronize(); torch.cuda.synchronize()
    assert mpc.launch_count == n0
    for t, w in zip((tq.servo, tq.force, tq.q_d, tq.tau_d, tq.grf), before):
        np.testing.assert_array_equal(t.cpu().numpy(), w)
    tq.force.zero_()
    assert rc() == 0
    mpc.synchronize()
    assert mpc.launch_count == n0 + 2
    assert not (tq.tau_d.cpu().numpy() == 7.0).any()
