"""Farm health counters (go1mpc_gait_stack_tick_clocked_health_async, go1mpc_servo_torque_tick_health_async, health_d of
go1mpc_farm_copy_async): per-robot solver outcomes counted on the device since each robot's reset.

- observational: a farm run through the health entries equals the same farm through the plain entries bit for bit (spread clocks,
  about 1 % device resets per period, restarts through the farm copy), at 16 and 2048 robots, as direct calls and as a replayed
  captured period graph; the health period launches exactly one kernel more; EVENTS holds the rows that grew in each period;
- planner and body rows against the oracle planner node in lock step (its step-timing tick replayed with diagnostics) and
  against the diag records of go1mpc_nlp_node_tick_batch + go1mpc_rt_node_tick_msgs_batch, cfg3 feedback gains, noisy foot feedback, a whole 700-period walk;
- spread clocks: each robot's counters equal a fresh aligned run's at the same clock;
- servo rows against the per-tick composition (distribution, force QP with diag, torque map, servo stack K = 1 update counts),
  K = 10 and K = 1, with NaN measured joints, NaN force commands and unreachable homing rows on some robots;
- restart at clock 0 through reset_d and a fresh bank column, snapshot / restore continuity, and argument refusal."""
import ctypes

import numpy as np
import pytest

import quadrupedal_loco_b200 as q
from tests.oracle_lib import P, StepCfg, StepDiag
from tests.test_gpu_farm_copy import GM, Robots, equal, idx
from tests.test_gpu_gait_stack import SERVO_SLOTS, planner_ticks
from tests.test_gpu_gait_stack_clocked import NH, K, Q0, servo_columns, staggered_inputs
from tests.test_gpu_servo_torque import WARM, YC, Chain, Torque, meas0, set_right_support, walked

pytestmark = pytest.mark.gpu

H = q.HEALTH_ROWS
STEP_LAMDA = (0.25, 0.001, 0.025, 0.001)      # cfg3's feedback-gain presets (bench.py)
BODY_LAMDA = (0.2, 0.001, 0.2, 0.001)


def health(B):
    import torch
    return torch.zeros(H, B, dtype=torch.int32, device="cuda")


def period(r, h=None, reset_d=None, restart=None, sensor_d=None, cmd_d=None, start_d=None, K_=K):
    """restore (restart = (bank, bank health or None, index_d)) or reset -> clocked tick -> torque tick, with health h or without."""
    mpc, f = r.mpc, r.f
    if restart is not None:
        bank, bh, index = restart
        d, s = r.cols(), bank.cols()
        if h is not None:
            d.health_d, s.health_d = h.data_ptr(), bh.data_ptr()
        mpc.farm_copy(NH, d, s, index, stream=r.stream)
    if reset_d is not None:
        rs = mpc.gait_stack_reset_struct(NH, None, f.clock, f.state, f.body_out, f.servo, Q0, reset_d=reset_d)
        mpc.gait_stack_reset_async(r.B, rs, r.stream)
    t = mpc.gait_stack_tick_clocked_struct(NH, None, f.clock, f.state, f.body_out, SERVO_SLOTS, f.rows_d, sensor_d=sensor_d,
                                           cmd_d=cmd_d, start_d=start_d)
    mpc.gait_stack_tick_clocked_async(r.B, t, r.stream, health_d=h)
    mpc.servo_torque_tick(r.B, K_, GM, 1.0, YC, f.state, f.servo, r.force, r.meas, f.q_d, r.tau_d, stream=r.stream,
                          reset_d=reset_d, health_d=h)


def spread_inputs(R, T, seed):
    """staggered_inputs on the device, with about 1 % extra resets per period and restarts from a bank every 50 periods."""
    I = staggered_inputs(R, T, seed)
    rng = np.random.Generator(np.random.Philox(seed + 1))
    flags = I["flags"] | (rng.random((T, R)) < 0.01).astype(np.int32)
    flags[0] = 0
    index = np.full((T, R), -1, np.int32)
    for j in range(25, T, 50):
        pick = rng.random(R) < 0.01
        pick[j % R] = True
        index[j, pick] = rng.integers(0, 4, pick.sum())
    import torch
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return dict(flags=dv(flags), index=dv(index), sensor=dv(I["sensor"]), cmd=dv(I["cmd"]), start=dv(I["start"]))


def grown_bits(new, old):
    import torch
    w = torch.tensor([1 << r for r in range(H - 1)], dtype=torch.int32, device=new.device)[:, None]
    return ((new[:H - 1] > old[:H - 1]).to(torch.int32) * w).sum(dim=0).to(torch.int32)


@pytest.mark.parametrize("R", [16, 2048])
def test_health_entries_change_no_output(mpc, oracle, R):
    """T = 200 periods, spread clocks, ~1 % device resets, restarts from a fresh bank: the health farm's every block, rows, q, tau
    equal the plain farm's, as direct calls and as a captured period graph; the health period launches one kernel more; EVENTS
    equals, every period, the rows that grew (from zero for the robots that restarted)."""
    import torch
    T = 200
    D = spread_inputs(R, T, 700 + R)
    servo, meas = servo_columns(oracle, R, 701 + R, jitter=False), meas0(R, 702 + R)
    s = torch.cuda.Stream()
    farms = {m: Robots(mpc, R, servo, meas, s.cuda_stream) for m in ("plain", "health", "graph")}
    hs = {m: health(R) for m in ("health", "graph")}
    bank = Robots(mpc, 4, servo[:, :4], meas[:, :4], s.cuda_stream)        # freshly reset robots: clock 0, default columns
    bank_h = health(4)
    bank_h.fill_(77)
    hist = {m: [torch.zeros(T, R, n, dtype=torch.float64, device="cuda") for n in (len(SERVO_SLOTS), 12 * K, 12 * K)] for m in farms}
    hh = torch.zeros(T + 1, H, R, dtype=torch.int32, device="cuda")
    clocks = torch.zeros(T, R, dtype=torch.int32, device="cuda")
    launches = {}
    # the graph farm's inputs, rewritten on the device before each replay
    cur = dict(flags=torch.zeros(R, dtype=torch.int32, device="cuda"), index=torch.full((R,), -1, dtype=torch.int32, device="cuda"),
               sensor=torch.zeros_like(D["sensor"][0]), cmd=torch.zeros_like(D["cmd"][0]), start=torch.zeros_like(D["start"][0]))

    def run(m, j, h, **kw):
        r = farms[m]
        n0 = mpc.launch_count
        period(r, h, reset_d=kw["flags"], restart=(bank, bank_h if h is not None else None, kw["index"]), sensor_d=kw["sensor"],
               cmd_d=kw["cmd"], start_d=kw["start"])
        launches.setdefault(m, set()).add(mpc.launch_count - n0)
        for a, t in zip(hist[m], (r.f.rows_d, r.f.q_d, r.tau_d)):
            a[j].copy_(t)

    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for j in range(T):
            kw = {k: D[k][j] for k in cur}
            run("plain", j, None, **kw)
            run("health", j, hs["health"], **kw)
            hh[j + 1].copy_(hs["health"]); clocks[j].copy_(farms["health"].f.clock)
        # warm-up of the graph farm on the same stream, then capture
        for k in cur:
            cur[k].copy_(D[k][0])
        run("graph", 0, hs["graph"], **cur)
    s.synchronize()
    ge = capture(mpc, s, lambda: period(farms["graph"], hs["graph"], reset_d=cur["flags"], restart=(bank, bank_h, cur["index"]),
                                        sensor_d=cur["sensor"], cmd_d=cur["cmd"], start_d=cur["start"]))
    try:
        with torch.cuda.stream(s):
            for j in range(1, T):
                for k in cur:
                    cur[k].copy_(D[k][j])
                mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, s.cuda_stream), "graph_launch")
                for a, t in zip(hist["graph"], (farms["graph"].f.rows_d, farms["graph"].f.q_d, farms["graph"].tau_d)):
                    a[j].copy_(t)
        s.synchronize()
    finally:
        mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
    torch.cuda.synchronize()
    for m in ("health", "graph"):
        for a, b in zip(hist[m], hist["plain"]):
            assert equal(a, b), m
        for a, b in zip(farms[m].buffers(), farms["plain"].buffers()):
            assert equal(a, b), m
    assert equal(hs["graph"], hs["health"])
    assert len(launches["plain"]) == 1 and launches["health"] == {launches["plain"].pop() + 1}
    # EVENTS: the rows that grew in the period, from zero for robots whose clock restarted
    for j in range(T):
        old = torch.where((clocks[j] == 1)[None, :], torch.zeros_like(hh[j]), hh[j])
        assert torch.equal(hh[j + 1][H - 1], grown_bits(hh[j + 1], old)), j
    fin = hs["health"].cpu().numpy()
    assert (fin[q.HEALTH_BODY_OK] > 0).any() and (fin[q.HEALTH_GRF_OK] > 0).any() and (fin[q.HEALTH_PLAN_OK] > 0).any()
    assert (D["index"] >= 0).sum() > 0 and D["flags"][1:].sum() > 0


def capture(mpc, s, body):
    mpc._check(mpc.lib.go1mpc_graph_capture_begin(mpc.h, s.cuda_stream), "capture_begin")
    body()
    ge = ctypes.c_void_p()
    mpc._check(mpc.lib.go1mpc_graph_capture_end(mpc.h, s.cuda_stream, ctypes.byref(ge)), "capture_end")
    return ge


class StepExt(ctypes.Structure):
    """orc_step_ext of oracle/go1_oracle.h."""
    _fields_ = [("ntdx", ctypes.c_int), ("zsc", ctypes.c_double * 12), ("zmpx", ctypes.c_double * 12), ("zmpy", ctypes.c_double * 12)]


N_TINT, STEP_STATE = 367, 202    # oracle/nlp_node.c: the node row of _t_int; the planner state is rows [0, 202) of the node


class OracleNode:
    """The oracle planner node (oracle/nlp_node.c) with cfg3's step gains.  tick runs orc_nlp_node_tick and returns the statuses of
    the SQP QPs its step-timing tick solved: the node calls orc_step_timing_tick_ext without diagnostics, so the same tick -- the
    node's t_int, its planner state before the call, the foot feedback x / y, a zero estimated state, flat ground (rt_nlp_gait) --
    is run again on a copy of that state with an orc_step_diag, and the copy must end bit-identical to the node's state."""

    def __init__(self, oracle):
        lib = self.lib = oracle.lib
        lib.orc_nlp_node_doubles.restype = ctypes.c_int
        self.cfg = (ctypes.c_double * 128)()              # orc_nlp_cfg, opaque except its leading orc_step_cfg
        lib.orc_nlp_cfg_default(self.cfg)
        sc = StepCfg.from_buffer(self.cfg)
        for i in range(4):
            sc.lamda[i] = STEP_LAMDA[i]
        self.node = np.zeros(lib.orc_nlp_node_doubles())
        lib.orc_nlp_node_default(self.cfg, P(self.node))
        self.out = np.zeros(100)

    def tick(self, w, start, rf, lf):
        before = self.node.copy()
        self.lib.orc_nlp_node_tick(self.cfg, P(self.node), int(w), int(start), P(np.ascontiguousarray(rf)), P(np.ascontiguousarray(lf)),
                                   P(self.out))
        t_int = int(self.node[N_TINT])
        if t_int == int(before[N_TINT]) or t_int < 1:      # _t_int grows on every walking call: no step-timing tick ran
            return []
        st = np.ascontiguousarray(before[:STEP_STATE])
        inp = np.zeros(21)                                 # orc_step_in: est[6] | rfoot_fb[2] | lfoot_fb[2] | comz, comaz, zsc, comvz0
        inp[6:8], inp[8:10] = rf[:2], lf[:2]
        d, ext, out38 = StepDiag(), StepExt(), np.zeros(38)
        self.lib.orc_step_timing_tick_ext(self.cfg, t_int, P(st), P(inp), P(out38), ctypes.byref(d), ctypes.byref(ext))
        assert np.array_equal(st.view(np.int64), self.node[:STEP_STATE].view(np.int64)), "replayed step tick differs from the node's"
        return [d.status[i] for i in range(d.n_solved)]


def noisy_sensors(T, R, seed):
    """Sensor rows [T][11][R]: control on, random body angles / rates, foot feedback around the stance with a per-robot noise
    amplitude (0 for every fourth robot)."""
    rng = np.random.Generator(np.random.Philox(seed))
    s = np.zeros((T, q.STACK_SENSOR_ROWS, R))
    s[:, 0] = 1.0
    s[:, 1:5] = rng.uniform(-0.03, 0.03, (T, 4, R))
    amp = (0.02 * (np.arange(R) % 4))[None, :]
    for base, y in ((5, 0.127), (8, -0.127)):
        s[:, base] = 3 * amp * rng.uniform(-1, 1, (T, R))
        s[:, base + 1] = np.where(amp > 0, y, 0.0) + amp * rng.uniform(-1, 1, (T, R))
        s[:, base + 2] = 0.2 * amp * rng.uniform(-1, 1, (T, R))
    return s


def split(status, axis):
    """OK / INFEASIBLE / FAILED counts of an int array of statuses (negative = no solve) over `axis`."""
    return [(status == 0).sum(axis=axis), (status == 2).sum(axis=axis), ((status >= 1) & (status != 2)).sum(axis=axis)]


def test_planner_and_body_counts_exact(oracle):
    """64 robots, aligned clocks, 700 periods, cfg3 gains: PLAN rows equal the oracle planner node run in lock step, BODY rows
    the body diag of go1mpc_nlp_node_tick_batch + go1mpc_rt_node_tick_msgs_batch, NONFINITE the periods with a non-finite rows_d
    row; every eighth robot never starts (its planner rows stay 0), every walking robot reaches PLAN_INFEASIBLE."""
    import torch
    R, T = 64, 700
    mpc = q.Go1Mpc(cfg={"lamda": BODY_LAMDA, "step": {"lamda": STEP_LAMDA}})
    try:
        dev = torch.device("cuda", 0)
        sensor = noisy_sensors(T, R, 800)
        start = np.ones((T, R), np.int32)
        start[:, ::8] = 0
        sd, std = torch.from_numpy(sensor).to(dev), torch.from_numpy(start).to(dev)
        col = mpc.gait_stack_default_state(NH)
        state = torch.from_numpy(np.repeat(col[:, None], R, axis=1).copy()).to(dev)
        body_out = torch.zeros(R, q.body_out_stride(NH), dtype=torch.float64, device=dev)
        rows_d = torch.zeros(R, len(SERVO_SLOTS), dtype=torch.float64, device=dev)
        clock, h = torch.zeros(R, dtype=torch.int32, device=dev), health(R)
        # the composition of the two node entries (tests/test_gpu_gait_stack.py), with the body diag
        nlp = torch.from_numpy(np.repeat(mpc.nlp_node_default_state()[:, None], R, axis=1).copy()).to(dev)
        rt = torch.from_numpy(np.repeat(mpc.rt_node_default_state(NH)[:, None], R, axis=1).copy()).to(dev)
        gait = torch.zeros(100, R, dtype=torch.float64, device=dev); traj = torch.zeros_like(gait)
        r2n = torch.zeros(25, R, dtype=torch.float64, device=dev); ctl = torch.zeros_like(r2n)
        body_in = torch.zeros(R, q.body_in_stride(NH), dtype=torch.float64, device=dev)
        body_out2 = torch.zeros_like(body_out)
        bdiag = torch.zeros(T, R, q.body_diag_stride(NH), dtype=torch.int32, device=dev)
        wd = torch.zeros(R, dtype=torch.int32, device=dev)
        ctl_slots = [0, 10, 11, 13, 14, 19, 20, 21, 22, 23, 24]
        hh = torch.zeros(T, H, R, dtype=torch.int32, device=dev)
        rows_hist = torch.zeros(T, R, len(SERVO_SLOTS), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
            for k in range(T):
                t = mpc.gait_stack_tick_clocked_struct(NH, None, clock, state, body_out, SERVO_SLOTS, rows_d, sensor_d=sd[k], start_d=std[k])
                mpc.gait_stack_tick_clocked_async(R, t, health_d=h)
                hh[k].copy_(h); rows_hist[k].copy_(rows_d)
                if planner_ticks(k):
                    wd += 1
                    mpc.nlp_node_tick(R, nlp, wd, gait, start_d=std[k], rfoot_fb_d=r2n[22:25], lfoot_fb_d=r2n[19:22])
                ctl[ctl_slots] = sd[k]
                mpc.rt_node_tick_msgs(NH, R, rt, gait, ctl, body_in, body_out2, traj, r2n, body_diag_d=bdiag[k])
        mpc.synchronize(); torch.cuda.synchronize()
        assert equal(body_out, body_out2)
        got = hh[-1].cpu().numpy()
        body = split(bdiag[:, :, 0].cpu().numpy(), 0)
        for i, row in enumerate((q.HEALTH_BODY_OK, q.HEALTH_BODY_INFEASIBLE, q.HEALTH_BODY_FAILED)):
            np.testing.assert_array_equal(got[row], body[i])
        # the oracle node in lock step, fed the foot feedback the previous fast tick forwarded
        plan = np.full((T, R, 8), -1)
        for r in range(R):
            node, w, fb = OracleNode(oracle), 0, np.zeros(6)
            for k in range(T):
                if planner_ticks(k):
                    w += 1
                    st = node.tick(w, start[k, r], fb[3:6].copy(), fb[0:3].copy())
                    plan[k, r, :len(st)] = st
                fb = sensor[k, 5:11, r]
        want = split(plan, (0, 2))
        for i, row in enumerate((q.HEALTH_PLAN_OK, q.HEALTH_PLAN_INFEASIBLE, q.HEALTH_PLAN_FAILED)):
            np.testing.assert_array_equal(got[row], want[i], err_msg=f"health row {row}")
        # the reference's 0 / 0 in a double-support phase with coinciding ZMP anchors leaves NaN in some result slots
        np.testing.assert_array_equal(got[q.HEALTH_NONFINITE], (~torch.isfinite(rows_hist)).any(dim=2).sum(dim=0).cpu().numpy())
        idle = np.arange(R) % 8 == 0
        assert (got[q.HEALTH_PLAN_INFEASIBLE, idle] == 0).all() and (got[q.HEALTH_PLAN_INFEASIBLE, ~idle] > 0).all()
        assert (got[q.HEALTH_PLAN_OK, ~idle] > 0).all()
        print(f"\nplanner INFEASIBLE per walking robot {got[q.HEALTH_PLAN_INFEASIBLE, ~idle].min()}..{got[q.HEALTH_PLAN_INFEASIBLE].max()}, "
              f"FAILED max {got[q.HEALTH_PLAN_FAILED].max()}; body OK max {got[q.HEALTH_BODY_OK].max()}, "
              f"BODY_INFEASIBLE total {got[q.HEALTH_BODY_INFEASIBLE].sum()}, BODY_FAILED total {got[q.HEALTH_BODY_FAILED].sum()}, "
              f"NONFINITE per robot {got[q.HEALTH_NONFINITE].min()}..{got[q.HEALTH_NONFINITE].max()} of {T}")
        # EVENTS of the clocked tick alone: the rows that grew in the call
        for k in range(1, T):
            assert torch.equal(hh[k][H - 1], grown_bits(hh[k], hh[k - 1])), k
    finally:
        mpc.close()


def test_spread_clock_counters_equal_fresh_runs(mpc, oracle):
    """Robots reset at their own periods (reset_d): each robot's counters at the end equal those of an aligned fresh run fed its
    inputs from its last reset on, read at the same clock."""
    import torch
    R, T = 256, 260
    I = staggered_inputs(R, T, 900)
    last = I["last"]
    servo, meas = servo_columns(oracle, R, 901, jitter=False), meas0(R, 902)
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    farm, ref = Robots(mpc, R, servo, meas), Robots(mpc, R, servo, meas)
    hf, hr = health(R), health(R)
    hist = torch.zeros(T, H, R, dtype=torch.int32, device="cuda")
    flags, sensor, cmd, start = dv(I["flags"]), dv(I["sensor"]), dv(I["cmd"]), dv(I["start"])
    rs, rc, rst = dv(I["ref_sensor"]), dv(I["ref_cmd"]), dv(I["ref_start"])
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        for k in range(T):
            period(farm, hf, reset_d=flags[k], sensor_d=sensor[k], cmd_d=cmd[k], start_d=start[k])
            period(ref, hr, sensor_d=rs[k], cmd_d=rc[k], start_d=rst[k])
            hist[k].copy_(hr)
    mpc.synchronize(); torch.cuda.synchronize()
    want = hist[torch.from_numpy(T - 1 - last).cuda(), :, torch.arange(R, device="cuda")].T
    assert torch.equal(hf[:H - 1], want[:H - 1])
    np.testing.assert_array_equal(farm.f.clock.cpu().numpy(), T - last)
    assert len(set(last % 5)) == 5 and (hf[q.HEALTH_GRF_OK] > 0).all()


def _iter_mpc(mpc, iters):
    """The handle with servo_stack_tick passing iters_d (the update counts of Chain's K = 1 servo stack calls)."""
    class M:
        def __getattr__(self, n):
            return getattr(mpc, n)

        def servo_stack_tick(self, *a, **kw):
            kw["iters_d"] = iters
            return mpc.servo_stack_tick(*a, **kw)
    return M()


@pytest.mark.parametrize("Kc", [10, 1])
def test_servo_counts_exact(mpc, oracle, Kc):
    """B = 512 on a walked gait stack, 4 periods of 10 ticks in calls of Kc ticks: GRF_OK / GRF_FAILED / GRF_FALLBACK / IK_CAP /
    NONFINITE equal the per-tick composition's force-QP diag, update counts and non-finite q / tau; EVENTS the rows that grew
    in each call.  NaN measured joints (robots 8i + 1, NONFINITE through the swing legs' torques: measured joints do not enter the
    QP), a NaN force command (8i + 3, GRF_FALLBACK every tick) and an FR homing row out of reach (8i + 5, IK_CAP every tick) drive
    the rows; the other robots stay at zero in GRF_FALLBACK and NONFINITE."""
    import torch
    B, T = 512, 4
    from tests.test_gpu_servo_stack import servo_state0, walk
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        st, sensor, start = walked(mpc, B, 71, T)
        gait = st.block(q.STACK_ROW_GAIT, 100)
        s0 = servo_state0(oracle, B, 73)
        m0 = meas0(B, 75)
        r = np.arange(B)
        m0[:12, r % 8 == 1] = np.nan
        s0[q.SERVO_ROW_HOMING + 2, r % 8 == 5] = -1.5                  # FR foot 1.5 m below the hip: out of reach
        tq = Torque(B, Kc, s0, m0)
        h = health(B)
        iters = torch.zeros(4, B, dtype=torch.int32, device="cuda")
        ch = Chain(_iter_mpc(mpc, iters), B, s0, m0)
        want = torch.zeros(H - 1, B, dtype=torch.int64, device="cuda")
        ev_bad = torch.zeros((), dtype=torch.int64, device="cuda")
        nan_cmd = torch.from_numpy(r % 8 == 3).cuda()
        for k in range(WARM, WARM + T):
            walk(st, sensor, start, k, k + 1)
            rs_old = set_right_support(gait, k)
            f_old = gait[15].clone()
            gait[15] = torch.where(nan_cmd, torch.full_like(f_old, float("nan")), f_old)
            for c in range(K // Kc):
                before = want.clone()
                h[H - 1].zero_()
                tq.call(mpc, st.state, GM, 1.0, health_d=h)
                for j in range(Kc):
                    q1, tau = ch.tick(st.state, GM, 1.0)
                    s_ = ch.diag[:, 0]
                    want[q.HEALTH_GRF_OK] += s_ == 0
                    want[q.HEALTH_GRF_FAILED] += s_ != 0
                    want[q.HEALTH_GRF_FALLBACK] += ch.diag[:, 6] == 0
                    want[q.HEALTH_IK_CAP] += (iters == 15).sum(dim=0)
                    want[q.HEALTH_NONFINITE] += (~torch.isfinite(q1)).any(dim=1) | (~torch.isfinite(tau)).any(dim=0)
                ev_bad += (h[H - 1] != grown_bits(want, before)).sum()
            gait[15] = f_old
            gait[99] = rs_old
    mpc.synchronize(); torch.cuda.synchronize()
    got = h[:H - 1].to(torch.int64)
    assert torch.equal(got, want)
    assert ev_bad.item() == 0
    g = got.cpu().numpy()
    quiet = (r % 8) % 2 == 0
    for row in (q.HEALTH_GRF_FALLBACK, q.HEALTH_NONFINITE):
        assert (g[row, quiet] == 0).all(), row
    assert (g[q.HEALTH_NONFINITE, r % 8 == 1] > 0).any() and (g[q.HEALTH_GRF_FALLBACK, r % 8 == 3] > 0).all()
    # the walked gait's leg IKs hit the 15-update cap now and then on every robot; an unreachable FR foot caps every tick
    assert (g[q.HEALTH_IK_CAP, r % 8 == 5] >= K * T).all() and g[q.HEALTH_IK_CAP, r % 8 == 5].min() > g[q.HEALTH_IK_CAP, quiet].max()
    print(f"\nIK_CAP per robot over {K * T} ticks: quiet robots {g[q.HEALTH_IK_CAP, quiet].min()}..{g[q.HEALTH_IK_CAP, quiet].max()}, "
          f"unreachable FR foot {g[q.HEALTH_IK_CAP, r % 8 == 5].min()}..{g[q.HEALTH_IK_CAP, r % 8 == 5].max()}; "
          f"GRF_FAILED total {g[q.HEALTH_GRF_FAILED].sum()}")
    assert (g[q.HEALTH_PLAN_OK:q.HEALTH_BODY_FAILED + 1] == 0).all()
    assert g[q.HEALTH_GRF_OK].sum() + g[q.HEALTH_GRF_FAILED].sum() == B * K * T


def test_restart_snapshot_and_restore(mpc, oracle):
    """Counters restart at clock 0 through reset_d and through a restore from a fresh bank column; a snapshot and restore with
    health on both sides continues counting bit-identically; a restore without health leaves the old counters."""
    import torch
    R, T = 64, 40
    D = spread_inputs(R, 2 * T, 950)
    servo, meas = servo_columns(oracle, R, 951, jitter=False), meas0(R, 952)
    a = Robots(mpc, R, servo, meas)
    ha = health(R)
    none = torch.full((R,), -1, dtype=torch.int32, device="cuda")
    zero = torch.zeros(R, dtype=torch.int32, device="cuda")
    feed = lambda j: dict(sensor_d=D["sensor"][j], cmd_d=D["cmd"][j], start_d=D["start"][j])
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        for j in range(T):
            period(a, ha, reset_d=zero, **feed(j))
        bank, hb = Robots(mpc, R, servo, meas), health(R)
        ident = idx(np.arange(R))
        period_copy = lambda d, dh, s, sh, index: mpc.farm_copy(NH, cols(d, dh), cols(s, sh), index)
        period_copy(bank, hb, a, ha, ident)                                     # snapshot at period T
        snap = ha.clone()
        for j in range(T, T + 10):
            period(a, ha, reset_d=zero, **feed(j))
        cont = ha.clone()
        b, hb2 = Robots(mpc, R, servo, meas), health(R)
        hb2.fill_(5)
        period_copy(b, hb2, bank, hb, ident)                                    # restore into other values
        restored = hb2.clone()
        for j in range(T, T + 10):
            period(b, hb2, reset_d=zero, **feed(j))
        # clock-0 restarts: reset robot 3, restore robot 9 from a fresh bank column
        fresh, hf = Robots(mpc, 1, servo[:, :1], meas[:, :1]), health(1)
        hf.fill_(55)                                                            # copied along, then zeroed by the clock-0 restart
        fl = torch.zeros(R, dtype=torch.int32, device="cuda"); fl[3] = 1
        ix = none.clone(); ix[9] = 0
        period(a, ha, restart=(fresh, hf, ix), reset_d=fl, **feed(T + 10))
        after = ha.clone(); clk = a.f.clock.clone()
        # a restore without health keeps the destination's counters
        keep = ha.clone()
        mpc.farm_copy(NH, a.cols(), bank.cols(), ident)
        kept = ha.clone()
    mpc.synchronize(); torch.cuda.synchronize()
    assert equal(restored, snap) and equal(hb2, cont)
    c = clk.cpu().numpy()
    assert c[3] == 1 and c[9] == 1 and (np.delete(c, [3, 9]) == T + 11).all()
    fr = after[:, [3, 9]].cpu().numpy()                                        # one period since the restart
    assert (fr[q.HEALTH_PLAN_OK:q.HEALTH_PLAN_FAILED + 1].sum(axis=0) <= 3).all()
    assert (fr[q.HEALTH_BODY_OK:q.HEALTH_BODY_FAILED + 1].sum(axis=0) <= 1).all()
    assert (fr[q.HEALTH_GRF_OK] + fr[q.HEALTH_GRF_FAILED] == K).all() and (fr[:H - 1] < 55).all()
    assert (after[q.HEALTH_GRF_OK, 0] + after[q.HEALTH_GRF_FAILED, 0]).item() == K * (T + 11)
    assert equal(kept, keep)


def cols(r, h):
    c = r.cols()
    c.health_d = h.data_ptr()
    return c


def test_health_rejects_bad_arguments(mpc, oracle):
    """Null, misaligned and overlapping health_d in both entries, and a health block on one side of a copy: GO1MPC_E_INVALID with
    the launch count unmoved and nothing written; valid calls then run."""
    import torch
    B = 64
    r = Robots(mpc, B, servo_columns(oracle, B, 990, jitter=True), meas0(B, 991))
    f = r.f
    h = health(B)
    sensor = torch.zeros(q.STACK_SENSOR_ROWS, B, dtype=torch.float64, device="cuda"); sensor[0] = 1.0
    reset = torch.zeros(B, dtype=torch.int32, device="cuda")
    grf, gdiag = torch.zeros(B, 16, dtype=torch.float64, device="cuda"), torch.zeros(B, 32, dtype=torch.int32, device="cuda")
    jac, fdes = torch.zeros(36, B, dtype=torch.float64, device="cuda"), torch.zeros(12, B, dtype=torch.float64, device="cuda")
    iters = torch.zeros(4, B, dtype=torch.int32, device="cuda")
    hp = h.data_ptr()

    def tick_rc(hd):
        t = mpc.gait_stack_tick_clocked_struct(NH, None, f.clock, f.state, f.body_out, SERVO_SLOTS, f.rows_d, sensor_d=sensor,
                                               start_d=reset)
        return mpc.lib.go1mpc_gait_stack_tick_clocked_health_async(mpc.h, B, ctypes.byref(t), hd, None)

    def torque_rc(hd):
        t = mpc.servo_torque_tick_struct(K, GM, 1.0, YC, f.state, f.servo, r.force, r.meas, f.q_d, r.tau_d, reset_d=reset,
                                         grf_d=grf, grf_diag_d=gdiag, jac_d=jac, foot_des_d=fdes, iters_d=iters)
        return mpc.lib.go1mpc_servo_torque_tick_health_async(mpc.h, B, ctypes.byref(t), hd, None)

    def copy_rc(dh, sh):
        d, s = r.cols(), r.cols()
        bank = Robots(mpc, B, servo_columns(oracle, B, 992, jitter=False), meas0(B, 993))
        s = bank.cols()
        d.health_d, s.health_d = dh, sh
        c = q.FarmCopy(NH, d, s, idx(np.arange(B)).data_ptr(), None)
        return mpc.lib.go1mpc_farm_copy_async(mpc.h, ctypes.byref(c), None), bank

    tick_cases = [None, hp + 2, f.state.data_ptr() + 8 * 100, f.body_out.data_ptr(), f.rows_d.data_ptr() + 8,
                  f.clock.data_ptr(), sensor.data_ptr() + 16, reset.data_ptr()]
    torque_cases = [None, hp + 1, f.state.data_ptr() + 8 * B * q.STACK_ROW_GAIT, f.servo.data_ptr(), r.force.data_ptr() + 8,
                    r.meas.data_ptr(), f.q_d.data_ptr(), r.tau_d.data_ptr() + 8 * 100, reset.data_ptr(), grf.data_ptr(),
                    gdiag.data_ptr(), jac.data_ptr(), fdes.data_ptr(), iters.data_ptr()]
    torch.cuda.synchronize()
    before = [t.clone() for t in r.buffers() + (f.rows_d, f.q_d, r.tau_d, h)]
    n0 = mpc.launch_count
    for hd in tick_cases:
        assert tick_rc(hd) == -1, hd
    for hd in torque_cases:
        assert torque_rc(hd) == -1, hd
    banks = []
    for dh, sh in ((hp, None), (None, health(B).data_ptr()), (hp + 2, health(B).data_ptr())):
        rc, bank = copy_rc(dh, sh)
        banks.append(bank)
        assert rc == -1, (dh, sh)
    mpc.synchronize(); torch.cuda.synchronize()
    assert mpc.launch_count == n0
    for a, b in zip(r.buffers() + (f.rows_d, f.q_d, r.tau_d, h), before):
        assert equal(a, b)
    assert tick_rc(hp) == 0 and torque_rc(hp) == 0
    mpc.synchronize()
    assert mpc.launch_count > n0 and (h[q.HEALTH_GRF_OK] + h[q.HEALTH_GRF_FAILED] == K).all()
