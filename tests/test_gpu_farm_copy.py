"""Farm column copy (go1mpc_farm_copy_async): whole robots -- gait stack column, body-MPC record, clock, servo column, force
column -- copied between farm-shaped buffer sets, the source column picked per destination by a device index.

- continuation: a farm snapshotted into a bank mid-walk and restored into a farm holding other values continues bit for bit
  (staggered clocks and resets, torque tick K = 10), at 16 robots (combined body kernel) and 2048 (three-launch body path);
- a permuted restore with permuted inputs gives the permuted outputs; one bank column forked into 1024 robots;
- a sparse restore (about 1 %) leaves every other column untouched, and every robot continues on its own timeline;
- restoring a bank column stored right after a reset equals the reset (with the torque tick's reset flag);
- bad indices keep their columns and are counted; one captured period graph (restore -> clocked tick -> torque tick) with the
  index rewritten on the device between replays; batch-size changes on one stream; argument refusal.
Every comparison is bit for bit: a mismatch would mean per-robot state outside the copied buffers."""
import ctypes

import numpy as np
import pytest

import quadrupedal_loco_b200 as q
from tests.test_gpu_gait_stack import SERVO_SLOTS
from tests.test_gpu_gait_stack_clocked import NH, K, Farm, bits, servo_columns, staggered_inputs
from tests.test_gpu_servo_stack import homing_feet
from tests.test_gpu_servo_torque import YC, meas0

pytestmark = pytest.mark.gpu

GM = 102


class Robots:
    """A farm on the clocked tick + torque tick: Farm's buffers plus the force state, measured joints and torques."""

    def __init__(self, mpc, B, servo, meas, stream=None):
        import torch
        dev = torch.device("cuda", 0)
        self.mpc, self.B, self.stream = mpc, B, stream
        self.f = Farm(mpc, B, servo, stream)
        self.force = torch.zeros(q.SERVO_FORCE_ROWS, B, dtype=torch.float64, device=dev)
        self.meas = torch.from_numpy(np.ascontiguousarray(meas)).to(dev)
        self.tau_d = torch.zeros(B, 12 * K, dtype=torch.float64, device=dev)

    def cols(self):
        f = self.f
        return self.mpc.farm_columns(self.B, f.state, f.body_out, f.clock, f.servo, self.force)

    def buffers(self):
        f = self.f
        return (f.state, f.body_out, f.clock, f.servo, self.force)

    def scramble(self, seed):
        """Other values in every block, so that anything a restore does not write shows."""
        import torch
        g = torch.Generator(device="cuda").manual_seed(seed)
        for t in (self.f.state, self.f.body_out, self.f.servo, self.force):
            t.normal_(generator=g)
        self.f.clock.random_(0, 1000, generator=g)

    def period(self, flags, sensor, cmd, start, reset=True):
        """reset -> clocked tick -> torque tick (K = 10) with the reset flags (host int32 [B]) also clearing the force state."""
        c = np.ascontiguousarray
        if reset:
            self.f.reset(c(flags))
        self.f.tick(c(sensor), cmd=c(cmd), start=c(start))
        self.mpc.servo_torque_tick(self.B, K, GM, 1.0, YC, self.f.state, self.f.servo, self.force, self.meas, self.f.q_d, self.tau_d,
                                   stream=self.stream, reset=c(flags) if reset else None)


def inputs_at(I, ks, cols):
    """One period's inputs for robots whose timeline stands at period ks[i], fed robot cols[i]'s inputs."""
    ks, cols = np.asarray(ks), np.asarray(cols)
    return I["flags"][ks, cols], I["sensor"][ks, :, cols].T, I["cmd"][ks, cols], I["start"][ks, cols]


def run(robots, I, ks0, cols, T, hist=None):
    """T periods, robot i fed at periods ks0[i], ks0[i] + 1, ...; returns [T][B][..] histories of rows, q, tau."""
    import torch
    B = robots.B
    if hist is None:
        hist = [torch.zeros(T, B, n, dtype=torch.float64, device="cuda") for n in (len(SERVO_SLOTS), 12 * K, 12 * K)]
    for j in range(T):
        robots.period(*inputs_at(I, np.asarray(ks0) + j, cols))
        for h, t in zip(hist, (robots.f.rows_d, robots.f.q_d, robots.tau_d)):
            h[j].copy_(t)
    return hist


def idx(a):
    import torch
    return torch.as_tensor(np.asarray(a, dtype=np.int32), device="cuda")


P_SNAP, T_CONT = 20, 40     # snapshot period; periods run after it (second resets of the staggered schedule fall inside)
_BASE = {}


def base_run(mpc, oracle, R):
    """Farm A on staggered inputs: bank = snapshot of every robot at period P_SNAP, then T_CONT more periods recorded.  Cached per R."""
    import torch
    if R in _BASE:
        return _BASE[R]
    I = staggered_inputs(R, P_SNAP + 2 * T_CONT, 300 + R)
    servo, meas = servo_columns(oracle, R, 301 + R, jitter=False), meas0(R, 302 + R)
    a = Robots(mpc, R, servo, meas)
    bank = Robots(mpc, R, servo, meas)
    bank.scramble(1)
    ident = np.arange(R)
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        run(a, I, np.zeros(R, int), ident, P_SNAP)
        mpc.farm_copy(NH, bank.cols(), a.cols(), idx(ident))
        hist = run(a, I, np.full(R, P_SNAP), ident, T_CONT)
    mpc.synchronize(); torch.cuda.synchronize()
    _BASE[R] = (I, servo, meas, a, bank, hist)
    return _BASE[R]


def equal(a, b):
    """Bit-for-bit equality of two tensors (float64 compared as bit patterns)."""
    import torch
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    return torch.equal(bits(a), bits(b)) if a.dtype == torch.float64 else torch.equal(a, b)


AOS = (False, True, True, False, False)      # per block of Robots.buffers(): robot index first (body records, clocks)


def pick(t, aos, cols):
    """Robot columns `cols` of one block."""
    return t[cols] if aos else t[:, cols]


@pytest.mark.parametrize("R", [16, 2048])
def test_continuation_from_snapshot(mpc, oracle, R):
    """Restoring the bank into a second farm whose buffers hold other values, and feeding it the same periods, reproduces the first
    farm's rows, joint targets and torques at every period and all its final buffers."""
    import torch
    I, servo, meas, a, bank, hist = base_run(mpc, oracle, R)
    b = Robots(mpc, R, servo, meas)
    b.scramble(2)
    ident = np.arange(R)
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        mpc.farm_copy(NH, b.cols(), bank.cols(), idx(ident))
        got = run(b, I, np.full(R, P_SNAP), ident, T_CONT)
    mpc.synchronize(); torch.cuda.synchronize()
    for h, w in zip(got, hist):
        assert equal(h, w)
    for x, y in zip(b.buffers(), a.buffers()):
        assert equal(x, y)
    assert (I["flags"][P_SNAP:P_SNAP + T_CONT].sum(axis=0) > 0).any()      # resets happen after the snapshot
    assert len(set(bank.f.clock.cpu().numpy() % 5)) == 5                   # staggered clocks in the bank
    assert (hist[2].abs().amax(dim=(1, 2)) > 0).all()


def test_permuted_restore_and_fork(mpc, oracle):
    """A restore with a random permutation, fed the permuted inputs, gives the permuted outputs; one bank column forked into 1024
    robots fed that robot's inputs all equal its continuation."""
    import torch
    R = 2048
    I, servo, meas, a, bank, hist = base_run(mpc, oracle, R)
    perm = np.random.default_rng(5).permutation(R)
    p = Robots(mpc, R, servo[:, perm], meas[:, perm])
    p.scramble(3)
    r0 = 77
    F = 1024
    fk = Robots(mpc, F, servo[:, [r0] * F], meas[:, [r0] * F])
    fk.scramble(4)
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        mpc.farm_copy(NH, p.cols(), bank.cols(), idx(perm))
        got = run(p, I, np.full(R, P_SNAP), perm, T_CONT)
        mpc.farm_copy(NH, fk.cols(), bank.cols(), idx(np.full(F, r0)))
        fgot = run(fk, I, np.full(F, P_SNAP), np.full(F, r0), T_CONT)
    mpc.synchronize(); torch.cuda.synchronize()
    pt = torch.from_numpy(perm).cuda()
    for h, w in zip(got, hist):
        assert equal(h, w[:, pt])
    for x, y, aos in zip(p.buffers(), a.buffers(), AOS):
        assert equal(x, pick(y, aos, pt))
    for h, w in zip(fgot, hist):
        assert equal(h, w[:, r0:r0 + 1].expand(-1, F, -1).contiguous())


def test_sparse_restore(mpc, oracle):
    """About 1 % of a walking farm restored from a bank taken T periods earlier, -1 elsewhere: the untouched columns of every block
    are bit-identical before and after the call; then the restored robots repeat their continuation from the bank's period and the
    others continue their own walk."""
    import torch
    R, T = 2048, 16
    I, servo, meas, a0, bank, hist = base_run(mpc, oracle, R)
    a = Robots(mpc, R, servo, meas)
    ident = np.arange(R)
    sel = np.random.default_rng(6).choice(R, 20, replace=False)
    index = np.full(R, -1); index[sel] = sel
    on = np.zeros(R, bool); on[sel] = True
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        mpc.farm_copy(NH, a.cols(), bank.cols(), idx(ident))                  # farm A at P_SNAP ...
        run(a, I, np.full(R, P_SNAP), ident, T)                                 # ... walked on to P_SNAP + T
        z = Robots(mpc, R, servo, meas)
        for x, y in zip(z.buffers(), a.buffers()):
            x.copy_(y)
        want_rest = run(a, I, np.full(R, P_SNAP + T), ident, T)                 # the untouched robots' continuation
    mpc.synchronize(); torch.cuda.synchronize()
    before = [t.clone() for t in z.buffers()]
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        mpc.farm_copy(NH, z.cols(), bank.cols(), idx(index))
    mpc.synchronize(); torch.cuda.synchronize()
    off = torch.from_numpy(~on).cuda()
    onm = torch.from_numpy(on).cuda()
    for x, y, bk, aos in zip(z.buffers(), before, bank.buffers(), AOS):
        assert equal(pick(x, aos, off), pick(y, aos, off)) and equal(pick(x, aos, onm), pick(bk, aos, onm))
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        got = run(z, I, np.where(on, P_SNAP, P_SNAP + T), ident, T)
    mpc.synchronize(); torch.cuda.synchronize()
    for h, w_rest, w_sel in zip(got, want_rest, hist):
        assert equal(h[:, off], w_rest[:, off])
        assert equal(h[:, onm], w_sel[:T, onm])


def test_restore_equals_reset(mpc, oracle):
    """A bank column stored right after go1mpc_gait_stack_reset_async (uniform homing, zero force state): restoring it into robots
    equals resetting them with the torque tick's reset flag, over the following periods."""
    import torch
    R, P, T = 256, 23, 30
    I = staggered_inputs(R, P + T, 17)
    servo = servo_columns(oracle, R, 18, jitter=True)
    servo[q.SERVO_ROW_HOMING:q.SERVO_ROW_HOMING + 12] = homing_feet(oracle)[:, None]
    meas = meas0(R, 19)
    ident = np.arange(R)
    fresh = Robots(mpc, 1, servo[:, :1], meas[:, :1])
    fresh.scramble(7)
    fresh.force.zero_()
    fresh.f.servo[q.SERVO_ROW_HOMING:q.SERVO_ROW_HOMING + 12] = torch.from_numpy(homing_feet(oracle)[:, None]).cuda()
    a = Robots(mpc, R, servo, meas)
    sel = np.zeros(R, np.int32); sel[3::9] = 1
    torch.cuda.synchronize()
    with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
        fresh.f.reset(np.ones(1, np.int32))
        bank = Robots(mpc, 1, servo[:, :1], meas[:, :1])
        mpc.farm_copy(NH, bank.cols(), fresh.cols(), idx([0]))
        run(a, I, np.zeros(R, int), ident, P)
        b = Robots(mpc, R, servo, meas)
        for x, y in zip(b.buffers(), a.buffers()):
            x.copy_(y)
        flags, sensor, cmd, start = inputs_at(I, np.full(R, P), ident)
        a.period(np.maximum(flags, sel), sensor, cmd, start)                   # reset + torque tick reset flag
        mpc.farm_copy(NH, b.cols(), bank.cols(), idx(np.where(sel == 1, 0, -1)))
        flags_b = np.where(sel == 1, 0, flags).astype(np.int32)
        b.period(flags_b, sensor, cmd, start)                                   # the restore instead of the reset
        ha = run(a, I, np.full(R, P + 1), ident, T - 1)
        hb = run(b, I, np.full(R, P + 1), ident, T - 1)
    mpc.synchronize(); torch.cuda.synchronize()
    for x, y in zip(ha, hb):
        assert equal(x, y)
    for x, y in zip(a.buffers(), b.buffers()):
        assert equal(x, y)
    assert (a.f.clock.cpu().numpy()[sel == 1] <= T).all()


def test_bad_indices_are_kept_and_counted(mpc, oracle):
    """Entries >= src.B or < -1 leave their destination columns untouched and add one each to bad_d; valid entries copy, -1 keeps."""
    import torch
    B, S = 64, 8
    servo, meas = servo_columns(oracle, B, 40, jitter=True), meas0(B, 41)
    dst, src = Robots(mpc, B, servo, meas), Robots(mpc, S, servo[:, :S], meas[:, :S])
    dst.scramble(8); src.scramble(9)
    index = np.full(B, -1, np.int64)
    index[0:8] = np.arange(S)[::-1]
    bad_vals = [S, S + 1, 1000, 2 ** 31 - 1, -2, -7, -(2 ** 31)]
    index[20:20 + len(bad_vals)] = bad_vals
    index[40] = 3
    bad = torch.full((1,), 5, dtype=torch.int32, device="cuda")
    index_d = idx(index)
    before = [t.clone() for t in dst.buffers()]
    torch.cuda.synchronize()
    mpc.farm_copy(NH, dst.cols(), src.cols(), index_d, bad_d=bad)
    mpc.synchronize()
    assert int(bad.item()) == 5 + len(bad_vals)
    ok = (index >= 0) & (index < S)
    kept = torch.from_numpy(~ok).cuda()
    took, srcs = torch.from_numpy(np.nonzero(ok)[0]).cuda(), torch.from_numpy(index[ok]).cuda()
    assert (~ok).sum() == len(bad_vals) + (index == -1).sum() and ok.sum() == 9
    for x, y, sv, aos in zip(dst.buffers(), before, src.buffers(), AOS):
        assert equal(pick(x, aos, kept), pick(y, aos, kept))
        assert equal(pick(x, aos, took), pick(sv, aos, srcs))


def test_one_graph_restore_tick_torque(mpc, oracle):
    """After warm-up, one period -- restore from an 8-column bank, clocked tick, torque tick K = 10 -- captured once and replayed
    30 times, a torch op rewriting index_d on the device and the pinned sensor buffer rewritten between replays, equals 30 direct
    periods bit for bit."""
    import torch
    R, S, W, N = 64, 8, 6, 30
    s = torch.cuda.Stream()
    I = staggered_inputs(R, 64, 90)      # 64 periods: the reset schedule reaches period 47; the test reads periods 0..W + N
    servo, meas = servo_columns(oracle, R, 91, jitter=False), meas0(R, 92)
    f = Robots(mpc, R, servo, meas, s.cuda_stream)
    bank = Robots(mpc, S, servo[:, :S], meas[:, :S], s.cuda_stream)
    rng = np.random.default_rng(93)
    table = np.where(rng.random((N + 1, R)) < 0.1, rng.integers(0, S, (N + 1, R)), -1).astype(np.int32)
    table_d = idx(table)
    index_d = torch.full((R,), -1, dtype=torch.int32, device="cuda")
    pin_sensor = torch.zeros(q.STACK_SENSOR_ROWS, R, dtype=torch.float64).pin_memory()
    ident = np.arange(R)
    hist = {m: [torch.zeros(N, R, n, dtype=torch.float64, device="cuda") for n in (len(SERVO_SLOTS), 12 * K, 12 * K)]
            for m in ("direct", "graph")}

    def period():
        mpc.farm_copy(NH, f.cols(), bank.cols(), index_d, stream=s.cuda_stream)
        f.f.tick(pin_sensor)
        mpc.servo_torque_tick(R, K, GM, 1.0, YC, f.f.state, f.f.servo, f.force, f.meas, f.f.q_d, f.tau_d, stream=s.cuda_stream)

    def load(k, j):
        s.synchronize()
        pin_sensor.copy_(torch.from_numpy(np.ascontiguousarray(I["sensor"][k])))
        with torch.cuda.stream(s):
            index_d.copy_(table_d[j])

    def record(m, j):
        with torch.cuda.stream(s):
            for h, t in zip(hist[m], (f.f.rows_d, f.f.q_d, f.tau_d)):
                h[j].copy_(t)

    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for k in range(W):
            f.period(*inputs_at(I, np.full(R, k), ident))
        mpc.farm_copy(NH, bank.cols(), f.cols(), idx(np.arange(S) * 5), stream=s.cuda_stream)
    s.synchronize()
    load(W, N)
    period()                                                               # warm-up of the period's own calls
    s.synchronize()
    snap0 = [t.clone() for t in f.buffers()]
    for j in range(N):
        load(W + 1 + j, j); period(); record("direct", j)
    s.synchronize()
    want = [t.clone() for t in f.buffers()]
    for t, t0 in zip(f.buffers(), snap0):
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
            load(W + 1 + j, j)
            mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, s.cuda_stream), "graph_launch")
            record("graph", j)
        s.synchronize()
    finally:
        mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
    for a, b in zip(hist["graph"], hist["direct"]):
        assert equal(a, b)
    for a, b in zip(f.buffers(), want):
        assert equal(a, b)
    assert (table[:N] >= 0).sum() > 50 and (hist["direct"][2].abs().amax(dim=(1, 2)) > 0).all()


def test_batch_size_changes_one_stream(mpc, oracle):
    """64 -> 3000 -> 64 destination columns on one stream, a fresh index each round: the 64-column copies equal the first 64
    columns of the 3000-column copies (no stale list or count of the larger call)."""
    import torch
    BS, BB, S = 64, 3000, 100
    s = torch.cuda.Stream()
    servo, meas = servo_columns(oracle, BB, 50, jitter=True), meas0(BB, 51)
    src = Robots(mpc, S, servo[:, :S], meas[:, :S])
    big = Robots(mpc, BB, servo, meas)
    small = Robots(mpc, BS, servo[:, :BS], meas[:, :BS])
    src.scramble(10); big.scramble(11)
    for x, y, aos in zip(small.buffers(), big.buffers(), AOS):
        x.copy_(pick(y, aos, slice(0, BS)))
    torch.cuda.synchronize()
    rng = np.random.default_rng(52)
    for rnd in range(4):
        index = np.where(rng.random(BB) < 0.5, rng.integers(0, S, BB), -1)
        with torch.cuda.stream(s):
            ib, isml = idx(index), idx(index[:BS])
        mpc.farm_copy(NH, small.cols(), src.cols(), isml, stream=s.cuda_stream)
        mpc.farm_copy(NH, big.cols(), src.cols(), ib, stream=s.cuda_stream)
        mpc.farm_copy(NH, small.cols(), src.cols(), isml, stream=s.cuda_stream)
        s.synchronize()
        for x, y, aos in zip(small.buffers(), big.buffers(), AOS):
            assert equal(x, pick(y, aos, slice(0, BS))), rnd
    took = np.nonzero(index >= 0)[0]
    assert equal(big.f.clock[took], src.f.clock[index[took]])


def test_farm_copy_rejects_bad_arguments(mpc, oracle):
    """Each bad argument returns its code, launches nothing and writes nothing to the destination."""
    import torch
    B, S = 64, 16
    servo, meas = servo_columns(oracle, B, 60, jitter=True), meas0(B, 61)
    dst, src = Robots(mpc, B, servo, meas), Robots(mpc, S, servo[:, :S], meas[:, :S])
    dst.scramble(12); src.scramble(13)
    index = idx(np.arange(B) % S)
    raw = torch.zeros(B * q.body_out_stride(NH) + 2, dtype=torch.float64, device="cuda")
    bad_body = raw[1:].data_ptr()
    D, Sr = dst.cols(), src.cols()

    def cols(F, **kw):
        d = {k: getattr(F, k) for k, _ in q.FarmColumns._fields_}
        d.update(kw)
        return q.FarmColumns(**d)

    def rc(nh=NH, dst_kw=None, src_kw=None, index_d=index.data_ptr()):
        c = q.FarmCopy(nh, cols(D, **(dst_kw or {})), cols(Sr, **(src_kw or {})), index_d, None)
        return mpc.lib.go1mpc_farm_copy_async(mpc.h, ctypes.byref(c), None)

    # a destination block inside the source's state, and a source block inside the destination's servo state
    inside_src = Sr.state_d + 8 * 1000
    cases = [
        (dict(dst_kw=dict(state_d=None)), -1), (dict(dst_kw=dict(body_out_d=None)), -1), (dict(src_kw=dict(state_d=None)), -1),
        (dict(src_kw=dict(body_out_d=None)), -1), (dict(index_d=None), -1),
        (dict(dst_kw=dict(clock_d=None)), -1), (dict(src_kw=dict(servo_state_d=None)), -1), (dict(dst_kw=dict(force_state_d=None)), -1),
        (dict(dst_kw=dict(body_out_d=bad_body)), -1), (dict(src_kw=dict(body_out_d=bad_body)), -1),
        (dict(src_kw=dict(B=0)), -1), (dict(dst_kw=dict(B=-1)), -1), (dict(src_kw=dict(B=-1)), -1),
        (dict(dst_kw=dict(force_state_d=inside_src)), -1), (dict(src_kw=dict(clock_d=D.servo_state_d + 8 * 70)), -1),
        (dict(src_kw=dict(state_d=D.state_d)), -1),
        (dict(nh=2), -4), (dict(nh=41), -4),
    ]
    torch.cuda.synchronize()
    before = [t.clone() for t in dst.buffers()]
    n0 = mpc.launch_count
    for kw, code in cases:
        assert rc(**kw) == code, kw
    assert mpc.lib.go1mpc_farm_copy_async(mpc.h, None, None) == -1
    assert rc(dst_kw=dict(B=0)) == 0 and rc(dst_kw=dict(B=0), src_kw=dict(B=0)) == 0    # dst.B = 0: a no-op
    mpc.synchronize(); torch.cuda.synchronize()
    assert mpc.launch_count == n0
    for x, y in zip(dst.buffers(), before):
        assert equal(x, y)
    assert rc() == 0                                                       # a valid call still works after the refusals
    mpc.synchronize()
    assert mpc.launch_count == n0 + 2
    assert equal(dst.f.clock, src.f.clock[torch.arange(B, device="cuda") % S])
