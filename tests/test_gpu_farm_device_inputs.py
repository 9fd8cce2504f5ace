"""Device-fed farm periods: the gait stack ticks' sensor_d / cmd_d / start_d, the reset's reset_d and the torque tick's reset_d,
read in place in stream order instead of being uploaded from host buffers.

- device inputs equal host inputs holding the same values, bit for bit, on both tick entries: staggered clocks, scripted sensor
  rows, a stop / restart command script, per-period reset flags on the reset and the torque tick, planner and non-planner
  periods, at 16 robots (combined body kernel) and 2048 (three-launch body path); one run mixes device and host inputs;
- a closed loop through a deterministic plant written as torch ops on the farm's stream (previous rows, joint targets and
  torques in; next sensors, measured joints, commands and reset flags out): 48 periods enqueued with one synchronisation at
  the end, as direct calls and as one captured period graph replayed with the plant between replays, equal the same loop
  synchronised every period and fed through pinned host buffers;
- restarts decided on the device through go1mpc_farm_copy_async with device sensors, replayed without a synchronisation, equal
  the synchronised host-fed loop;
- argument refusal: both or neither of a pair, misaligned device inputs, device inputs overlapping a block the call writes."""
import ctypes

import numpy as np
import pytest

import quadrupedal_loco_b200 as q
from tests.test_gpu_farm_copy import GM, Robots, equal, idx
from tests.test_gpu_gait_stack import SERVO_SLOTS, Stack, planner_ticks, scripted_inputs
from tests.test_gpu_gait_stack_clocked import NH, K, Q0, servo_columns, staggered_inputs
from tests.test_gpu_servo_torque import YC, meas0

pytestmark = pytest.mark.gpu


def cmd_script(T, R):
    """Planner commands [T][R] int32: stops (1), walk-again commands (2) and values that are no command (5), at periods that
    fall on and off each robot's planner periods."""
    cmd = np.zeros((T, R), np.int32)
    r = np.arange(R)
    cmd[10 + r % 13, r] = np.where(r % 3 == 0, 1, 0)
    cmd[30 + r % 11, r] = np.where(r % 6 == 0, 2, 0)
    cmd[20, r % 9 == 4] = 5
    return cmd


def to_device(**arrays):
    import torch
    return {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in arrays.items()}


def period(r, reset=None, reset_d=None, sensor=None, sensor_d=None, cmd=None, cmd_d=None, start=None, start_d=None,
           torque_reset=None, torque_reset_d=None, restart=None):
    """One farm period on Robots r: reset (or a restart through farm_copy: (bank, index_d)) -> clocked tick -> torque tick K = 10,
    each input from a host or a device buffer as given."""
    mpc, f = r.mpc, r.f
    if restart is not None:
        mpc.farm_copy(NH, r.cols(), restart[0].cols(), restart[1], stream=r.stream)
    elif reset is not None or reset_d is not None:
        rs = mpc.gait_stack_reset_struct(NH, reset, f.clock, f.state, f.body_out, f.servo, Q0, reset_d=reset_d)
        mpc.gait_stack_reset_async(r.B, rs, r.stream)
    t = mpc.gait_stack_tick_clocked_struct(NH, sensor, f.clock, f.state, f.body_out, SERVO_SLOTS, f.rows_d, cmd=cmd, start=start,
                                           sensor_d=sensor_d, cmd_d=cmd_d, start_d=start_d)
    mpc.gait_stack_tick_clocked_async(r.B, t, r.stream)
    mpc.servo_torque_tick(r.B, K, GM, 1.0, YC, f.state, f.servo, r.force, r.meas, f.q_d, r.tau_d, stream=r.stream,
                          reset=torque_reset, reset_d=torque_reset_d)


def new_hist(T, B):
    import torch
    return [torch.zeros(T, B, n, dtype=torch.float64, device="cuda") for n in (len(SERVO_SLOTS), 12 * K, 12 * K)]


def record(hist, r, j):
    for h, t in zip(hist, (r.f.rows_d, r.f.q_d, r.tau_d)):
        h[j].copy_(t)


@pytest.mark.parametrize("R", [16, 2048])
def test_clocked_device_inputs_equal_host_inputs(mpc, oracle, R):
    """Staggered clocks and resets, scripted sensors and commands: a farm fed every input from device buffers, and one mixing
    device sensors and start flags with host commands and reset flags, equal the host-fed farm in every period's rows, joint
    targets and torques and in the final state, body records, clocks, servo and force columns."""
    import torch
    T = 60
    I = staggered_inputs(R, T, 500 + R)
    cmd = cmd_script(T, R)
    servo, meas = servo_columns(oracle, R, 501 + R, jitter=False), meas0(R, 502 + R)
    D = to_device(sensor=I["sensor"], cmd=cmd, start=I["start"], flags=I["flags"])
    farms = {m: Robots(mpc, R, servo, meas) for m in ("host", "device", "mixed")}
    hist = {m: new_hist(T, R) for m in farms}
    c = np.ascontiguousarray
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        for k in range(T):
            fl, se, cm, st = c(I["flags"][k]), c(I["sensor"][k]), c(cmd[k]), c(I["start"][k])
            period(farms["host"], reset=fl, sensor=se, cmd=cm, start=st, torque_reset=fl)
            period(farms["device"], reset_d=D["flags"][k], sensor_d=D["sensor"][k], cmd_d=D["cmd"][k], start_d=D["start"][k],
                   torque_reset_d=D["flags"][k])
            period(farms["mixed"], reset=fl, sensor_d=D["sensor"][k], cmd=cm, start_d=D["start"][k], torque_reset_d=D["flags"][k])
            for m in farms:
                record(hist[m], farms[m], k)
    mpc.synchronize(); torch.cuda.synchronize()
    for m in ("device", "mixed"):
        for a, b in zip(hist[m], hist["host"]):
            assert equal(a, b), m
        for a, b in zip(farms[m].buffers(), farms["host"].buffers()):
            assert equal(a, b), m
    clock = farms["host"].f.clock.cpu().numpy()
    assert I["flags"][1:].sum() > 0 and len(set(clock % 5)) >= 3
    assert (cmd == 1).any() and (cmd == 2).any() and (I["start"] == 0).any()
    assert hist["host"][2].abs().amax() > 0


@pytest.mark.parametrize("R", [16, 2048])
def test_host_schedule_device_inputs_equal_host_inputs(mpc, R):
    """go1mpc_gait_stack_tick_host_async on the reference's schedule (planner and non-planner periods): device sensor, command
    and start buffers give the host buffers' rows, state and body records bit for bit."""
    import torch
    T = 60
    sensor, _, start = scripted_inputs(T, R, 520 + R)
    cmd = cmd_script(T, R)
    D = to_device(sensor=sensor, cmd=cmd, start=start)
    host, dev = Stack(mpc, NH, R, SERVO_SLOTS), Stack(mpc, NH, R, SERVO_SLOTS)
    rows = {m: torch.zeros(T, R, len(SERVO_SLOTS), dtype=torch.float64, device="cuda") for m in ("host", "device")}
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        for k in range(T):
            pl = planner_ticks(k)
            host.tick(pl, sensor[k], cmd=np.ascontiguousarray(cmd[k]), start=np.ascontiguousarray(start[k]))
            t = mpc.gait_stack_tick_struct(NH, pl, None, dev.state, dev.body_out, SERVO_SLOTS, dev.rows_d, sensor_d=D["sensor"][k],
                                           cmd_d=D["cmd"][k], start_d=D["start"][k])
            mpc.gait_stack_tick_host_async(R, t)
            rows["host"][k].copy_(host.rows_d); rows["device"][k].copy_(dev.rows_d)
    mpc.synchronize(); torch.cuda.synchronize()
    assert equal(rows["device"], rows["host"])
    assert equal(dev.state, host.state) and equal(dev.body_out, host.body_out)
    assert any(planner_ticks(k) for k in range(T)) and not all(planner_ticks(k) for k in range(T))


# ---- the closed loop: a deterministic plant on the farm's stream
FEET = np.array([0.0, 0.127, 0.0, 0.0, -0.127, 0.0])     # nominal left / right foot xyz of the sensor rows


class Loop:
    """A farm closed through the plant: Robots' buffers, the plant's outputs (device) and restart bookkeeping."""

    def __init__(self, mpc, R, servo, meas, stream, S=1):
        import torch
        dev = torch.device("cuda", 0)
        self.r = Robots(mpc, R, servo, meas, stream)
        self.r.f.q_d.copy_(torch.from_numpy(np.tile(Q0, K)).to(dev).expand(R, -1))     # the previous joint targets of period 0
        self.sensor = torch.zeros(q.STACK_SENSOR_ROWS, R, dtype=torch.float64, device=dev)
        self.cmd = torch.zeros(R, dtype=torch.int32, device=dev)
        self.start = torch.ones(R, dtype=torch.int32, device=dev)
        self.reset = torch.zeros(R, dtype=torch.int32, device=dev)
        self.index = torch.full((R,), -1, dtype=torch.int32, device=dev)
        self.S, self.ar = S, torch.arange(R, dtype=torch.int32, device=dev)
        self.feet = torch.from_numpy(FEET).to(dev)[:, None]

    def plant(self, j):
        """The previous period's rows, joint targets and torques -> this period's sensor rows, measured joints, commands, reset
        flags (a robot resets when the fractional part of 1000 x its summed last-tick |torque| is below 0.02) and restart index
        (the reset robots restart from bank column (robot + j) mod S)."""
        import torch
        f = self.r.f
        tau, qd = self.r.tau_d[:, 12 * (K - 1):], f.q_d[:, 12 * (K - 1):]
        self.sensor[0] = 1.0
        self.sensor[1:5] = 0.02 * torch.tanh(tau[:, :4]).T
        self.sensor[5:11] = self.feet + 0.01 * torch.tanh(f.rows_d[:, 3:9]).T
        self.r.meas[:12] = (qd + 0.001 * torch.tanh(tau)).T
        self.r.meas[12:] = 0.1 * torch.tanh(tau).T
        x = tau.abs().sum(dim=1) * 1000
        flag = (x - x.floor()) < 0.02
        self.reset.copy_(flag.to(torch.int32))
        self.index.copy_(torch.where(flag, (self.ar + j) % self.S, -1).to(torch.int32))
        y = qd.abs().sum(dim=1) * 100
        fy = y - y.floor()
        self.cmd.copy_(torch.where(fy < 0.03, 1, torch.where(fy < 0.06, 2, 0)).to(torch.int32))

    def device_period(self, restart_bank=None):
        if restart_bank is None:
            period(self.r, reset_d=self.reset, sensor_d=self.sensor, cmd_d=self.cmd, start_d=self.start, torque_reset_d=self.reset)
        else:
            period(self.r, sensor_d=self.sensor, cmd_d=self.cmd, start_d=self.start, restart=(restart_bank, self.index))


class Pinned:
    """Pinned host copies of a Loop's plant outputs, for the host-fed reference."""

    def __init__(self, R):
        import torch
        self.sensor = torch.zeros(q.STACK_SENSOR_ROWS, R, dtype=torch.float64).pin_memory()
        self.cmd = torch.zeros(R, dtype=torch.int32).pin_memory()
        self.start = torch.ones(R, dtype=torch.int32).pin_memory()
        self.reset = torch.zeros(R, dtype=torch.int32).pin_memory()

    def load(self, L):
        self.sensor.copy_(L.sensor); self.cmd.copy_(L.cmd); self.reset.copy_(L.reset)


def capture(mpc, s, body):
    mpc._check(mpc.lib.go1mpc_graph_capture_begin(mpc.h, s.cuda_stream), "capture_begin")
    body()
    ge = ctypes.c_void_p()
    mpc._check(mpc.lib.go1mpc_graph_capture_end(mpc.h, s.cuda_stream, ctypes.byref(ge)), "capture_end")
    return ge


def test_closed_loop_without_host_round_trip(mpc, oracle):
    """P = 48 periods of plant -> reset -> clocked tick -> torque tick, every input on the device: (a) direct calls and (b) one
    captured period graph replayed with the plant enqueued between replays, each with one synchronisation at the end, equal (c)
    the loop synchronised every period with the plant's outputs copied into pinned buffers and the host-fed entries called."""
    import torch
    R, P = 1024, 48
    s = torch.cuda.Stream()
    servo, meas = servo_columns(oracle, R, 540, jitter=False), meas0(R, 541)
    loops = {m: Loop(mpc, R, servo, meas, s.cuda_stream) for m in ("direct", "graph", "host")}
    hist = {m: new_hist(P, R) for m in loops}
    resets = {m: torch.zeros(P, R, dtype=torch.int32, device="cuda") for m in loops}
    pin = Pinned(R)
    torch.cuda.synchronize()
    L = loops["direct"]
    with torch.cuda.stream(s):
        for j in range(P):
            L.plant(j); L.device_period(); record(hist["direct"], L.r, j); resets["direct"][j].copy_(L.reset)
    s.synchronize()                                                        # (a): the only synchronisation
    L = loops["graph"]
    ge = capture(mpc, s, L.device_period)                                  # the entries were warmed up on s by (a)
    try:
        with torch.cuda.stream(s):
            for j in range(P):
                L.plant(j)
                mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, s.cuda_stream), "graph_launch")
                record(hist["graph"], L.r, j); resets["graph"][j].copy_(L.reset)
        s.synchronize()                                                    # (b): the only synchronisation
    finally:
        mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
    L = loops["host"]
    for j in range(P):
        with torch.cuda.stream(s):
            L.plant(j)
        s.synchronize()
        pin.load(L)
        with torch.cuda.stream(s):
            period(L.r, reset=pin.reset, sensor=pin.sensor, cmd=pin.cmd, start=pin.start, torque_reset=pin.reset)
            record(hist["host"], L.r, j); resets["host"][j].copy_(L.reset)
    s.synchronize(); torch.cuda.synchronize()
    for m in ("direct", "graph"):
        for a, b in zip(hist[m], hist["host"]):
            assert equal(a, b), m
        for a, b in zip(loops[m].r.buffers(), loops["host"].r.buffers()):
            assert equal(a, b), m
        assert equal(resets[m], resets["host"]), m
    n = resets["host"][1:].sum(dim=1).cpu().numpy()
    assert n.sum() > 0 and (n < R).all()                                   # resets inside the window, never all robots
    assert hist["host"][2].abs().amax() > 0


def test_device_restart_with_device_sensors(mpc, oracle):
    """Restarts decided on the device: the plant writes restart_idx_d, and a captured period restore -> clocked tick -> torque
    tick fed device sensors and commands is replayed P = 40 times with no synchronisation; it equals the synchronised loop fed
    pinned host sensors and commands."""
    import torch
    R, S, W, P = 512, 8, 6, 40
    s = torch.cuda.Stream()
    servo, meas = servo_columns(oracle, R, 560, jitter=False), meas0(R, 561)
    loops = {m: Loop(mpc, R, servo, meas, s.cuda_stream, S) for m in ("graph", "host")}
    bank = Robots(mpc, S, servo[:, :S], meas[:, :S], s.cuda_stream)
    hist = {m: new_hist(P, R) for m in loops}
    pin = Pinned(R)
    keep = torch.full((R,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for L in loops.values():                                           # the same W warm-up periods on both farms
            mpc.farm_copy(NH, L.r.cols(), bank.cols(), keep, stream=s.cuda_stream)     # warms the restore's workspace up
            for j in range(W):
                L.plant(j); L.device_period()
        mpc.farm_copy(NH, bank.cols(), loops["graph"].r.cols(), idx(np.arange(S) * 37), stream=s.cuda_stream)
    s.synchronize()
    L = loops["graph"]
    ge = capture(mpc, s, lambda: L.device_period(restart_bank=bank))
    restarts = torch.zeros(P, dtype=torch.int64, device="cuda")
    try:
        with torch.cuda.stream(s):
            for j in range(P):
                L.plant(W + j)
                mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, s.cuda_stream), "graph_launch")
                record(hist["graph"], L.r, j); restarts[j] = (L.index >= 0).sum()
        s.synchronize()                                                    # the only synchronisation of the replays
    finally:
        mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
    L = loops["host"]
    for j in range(P):
        with torch.cuda.stream(s):
            L.plant(W + j)
        s.synchronize()
        pin.load(L)
        with torch.cuda.stream(s):
            period(L.r, sensor=pin.sensor, cmd=pin.cmd, start=pin.start, restart=(bank, L.index))
            record(hist["host"], L.r, j)
    s.synchronize(); torch.cuda.synchronize()
    for a, b in zip(hist["graph"], hist["host"]):
        assert equal(a, b)
    for a, b in zip(loops["graph"].r.buffers(), loops["host"].r.buffers()):
        assert equal(a, b)
    n = restarts.cpu().numpy()
    assert n.sum() > 0 and (n < R).all()


def test_device_inputs_reject_bad_arguments(mpc, oracle):
    """Both or neither of each pair, misaligned device inputs, and device inputs overlapping a block the call writes: each call
    returns GO1MPC_E_INVALID, launches nothing and writes nothing; valid device-fed calls then run."""
    import torch
    B = 64
    r = Robots(mpc, B, servo_columns(oracle, B, 580, jitter=True), meas0(B, 581))
    f = r.f
    D = to_device(sensor=scripted_inputs(1, B, 582)[0][0], cmd=np.zeros(B, np.int32), start=np.ones(B, np.int32),
                  flags=(np.arange(B) % 3 == 0).astype(np.int32))
    sensor_h = np.ascontiguousarray(D["sensor"].cpu().numpy())
    flags_h = np.ascontiguousarray(D["flags"].cpu().numpy())
    cmd_h = np.zeros(B, np.int32)
    f.state.add_(1.0)                                                      # not the default column: a stray reset would show
    f.clock.fill_(7)
    r.force.fill_(0.5)
    sp, cp, stp, fp = (D[k].data_ptr() for k in ("sensor", "cmd", "start", "flags"))
    state_bytes = f.state.numel() * 8

    def tick_rc(entry="clocked", **kw):
        a = dict(sensor=None, sensor_d=sp, cmd_d=cp, start_d=stp); a.update(kw)
        if entry == "clocked":
            t = mpc.gait_stack_tick_clocked_struct(NH, a.pop("sensor"), f.clock, f.state, f.body_out, SERVO_SLOTS, f.rows_d, **a)
            return mpc.lib.go1mpc_gait_stack_tick_clocked_async(mpc.h, B, ctypes.byref(t), None)
        t = mpc.gait_stack_tick_struct(NH, True, a.pop("sensor"), f.state, f.body_out, SERVO_SLOTS, f.rows_d, **a)
        return mpc.lib.go1mpc_gait_stack_tick_host_async(mpc.h, B, ctypes.byref(t), None)

    def reset_rc(reset=None, reset_d=fp):
        rs = mpc.gait_stack_reset_struct(NH, reset, f.clock, f.state, f.body_out, f.servo, Q0, reset_d=reset_d)
        return mpc.lib.go1mpc_gait_stack_reset_async(mpc.h, B, ctypes.byref(rs), None)

    def torque_rc(**kw):
        t = mpc.servo_torque_tick_struct(K, GM, 1.0, YC, f.state, f.servo, r.force, r.meas, f.q_d, r.tau_d, **kw)
        return mpc.lib.go1mpc_servo_torque_tick_async(mpc.h, B, ctypes.byref(t), None)

    tick_cases = [
        dict(sensor=sensor_h), dict(sensor_d=None), dict(cmd=cmd_h), dict(start=np.ones(B, np.int32)),
        dict(sensor_d=sp + 4), dict(cmd_d=cp + 2), dict(start_d=stp + 1),
        dict(sensor_d=f.state.data_ptr() + 8 * 1000), dict(sensor_d=f.state.data_ptr() + state_bytes - 8),
        dict(sensor_d=f.rows_d.data_ptr()), dict(sensor_d=f.body_out.data_ptr() + 16), dict(cmd_d=f.clock.data_ptr()),
        dict(start_d=f.state.data_ptr() + 4 * 7),
    ]
    host_tick_cases = [dict(sensor=sensor_h), dict(sensor_d=None), dict(cmd=cmd_h), dict(sensor_d=f.state.data_ptr() + 8 * 64),
                       dict(start_d=f.rows_d.data_ptr() + 4)]
    reset_cases = [
        dict(reset=flags_h), dict(reset_d=None), dict(reset_d=fp + 2), dict(reset_d=f.clock.data_ptr()),
        dict(reset_d=f.clock.data_ptr() + 4 * (B - 1)), dict(reset_d=f.servo.data_ptr() + 8 * B * 30), dict(reset_d=f.state.data_ptr()),
        dict(reset_d=f.body_out.data_ptr() + 8),
    ]
    torque_cases = [
        dict(reset=flags_h, reset_d=fp), dict(reset_d=fp + 1), dict(reset_d=r.force.data_ptr() + 8 * 5),
        dict(reset_d=f.servo.data_ptr()), dict(reset_d=f.q_d.data_ptr() + 8 * B), dict(reset_d=r.tau_d.data_ptr() + 4),
    ]
    torch.cuda.synchronize()
    bufs = r.buffers() + (f.rows_d, f.q_d, r.tau_d)
    before = [t.clone() for t in bufs]
    n0 = mpc.launch_count
    for kw in tick_cases:
        assert tick_rc(**kw) == -1, kw
    for kw in host_tick_cases:
        assert tick_rc("host", **kw) == -1, kw
    for kw in reset_cases:
        assert reset_rc(**kw) == -1, kw
    for kw in torque_cases:
        assert torque_rc(**kw) == -1, kw
    mpc.synchronize(); torch.cuda.synchronize()
    assert mpc.launch_count == n0
    for a, b in zip(bufs, before):
        assert equal(a, b)
    # valid device-fed calls run after the refusals
    assert reset_rc() == 0 and tick_rc() == 0 and torque_rc(reset_d=fp) == 0
    mpc.synchronize()
    assert mpc.launch_count > n0
    ck = f.clock.cpu().numpy()
    assert (ck[flags_h != 0] == 1).all() and (ck[flags_h == 0] == 8).all()
