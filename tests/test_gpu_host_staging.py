"""Host-buffer entries against their device-pointer forms.

Every synchronous *_host entry and the three pipelined lane entries stage host buffers through the handle's device
buffers.  On one handle, at B = 1, 37, 1000 and 37 again (growth, then reuse of the staging), each must return what the
device form returns on the same inputs, bit for bit, with and without its optional buffers.  A handle serves at most
256 distinct streams: the call that would bring in a 257th fails and enqueues nothing."""
import ctypes

import numpy as np
import pytest

import quadrupedal_loco_b200 as q
from quadrupedal_loco_b200 import synth
from tests.test_grf import grf_inputs, tau_inputs

pytestmark = pytest.mark.gpu

SIZES = (1, 37, 1000, 37)
NH = 10
SENTINELS = {np.float64: (-1.2345678901234567e300, 7.654321098765432e-300), np.int32: (-123456789, 987654321)}


class Buf:
    """One pointer argument.  kind: "in" (read), "inout" (read and written), "out" (written: compared where the device
    form writes it), "dev" (a device buffer in both forms, read and written).  optional: passed as NULL in the run
    without optional buffers."""

    def __init__(self, kind, data=None, shape=None, dtype=np.float64, optional=False, dev_shape=None):
        self.kind, self.optional = kind, optional
        self.data = None if data is None else np.ascontiguousarray(data)
        self.shape = self.data.shape if data is not None else shape
        self.dtype = self.data.dtype.type if data is not None else dtype
        self.dev_shape = dev_shape or self.shape


def soa(a):
    return np.ascontiguousarray(np.asarray(a).reshape(len(a), -1).T)


def cleared(a):
    """A device result used as the next entry's input: elements the kernel left at the sentinel become 0."""
    a = a.copy()
    a[a == SENTINELS[a.dtype.type][0]] = 0
    return a


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64) if a.dtype == np.float64 else a.view(np.int32)


def run_device(mpc, host_name, dev_name, args, dev_args, fill, use_optional):
    """The device form; outputs start as the sentinel `fill` (0 or 1).  Returns the buffers as numpy arrays."""
    import torch
    res, ptrs = {}, []
    for k, a in enumerate(args):
        if not isinstance(a, Buf):
            ptrs.append(a)
            continue
        if a.optional and not use_optional:
            ptrs.append(None)
            continue
        if a.kind in ("in", "inout", "dev"):
            t = torch.from_numpy(a.data.copy()).cuda()
        else:
            t = torch.full(a.dev_shape, SENTINELS[a.dtype][fill], dtype=torch.from_numpy(np.zeros(1, a.dtype)).dtype, device="cuda")
        res[k] = t
        ptrs.append(t.data_ptr())
    torch.cuda.synchronize()
    rc = getattr(mpc.lib, dev_name)(mpc.h, *dev_args(ptrs))
    assert rc == 0, f"{dev_name}: {mpc.lib.go1mpc_last_error(mpc.h).decode()}"
    mpc.synchronize()
    torch.cuda.synchronize()
    return {k: t.cpu().numpy() for k, t in res.items()}


def host_entry(mpc, name):
    if name == "go1mpc_foot_trajectory_stop_batch_host":
        # binding.py declares this entry with the device form's trailing stream argument, one more than it takes
        return ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int, *[ctypes.c_void_p] * 8)((name, mpc.lib))
    return getattr(mpc.lib, name)


def run_host(mpc, host_name, args, use_optional, lane):
    import torch
    res, ptrs, keep = {}, [], []
    for k, a in enumerate(args):
        if not isinstance(a, Buf):
            ptrs.append(a)
            continue
        if a.optional and not use_optional:
            ptrs.append(None)
            continue
        if a.kind == "dev":
            t = torch.from_numpy(a.data.copy()).cuda()
            keep.append((k, t))
            ptrs.append(t.data_ptr())
            continue
        h = a.data.copy() if a.kind in ("in", "inout") else np.full(a.shape, SENTINELS[a.dtype][0], a.dtype)
        res[k] = h
        ptrs.append(h.ctypes.data)
    torch.cuda.synchronize()
    rc = host_entry(mpc, host_name)(mpc.h, *ptrs)
    assert rc == 0, f"{host_name}: {mpc.lib.go1mpc_last_error(mpc.h).decode()}"
    if lane:
        mpc.synchronize()
    torch.cuda.synchronize()
    for k, t in keep:
        res[k] = t.cpu().numpy()
    return res


def check_entry(mpc, spec, lane=False):
    host_name, dev_name, args, dev_args = spec
    for use_optional in (True, False):
        d0 = run_device(mpc, host_name, dev_name, args, dev_args, 0, use_optional)
        d1 = run_device(mpc, host_name, dev_name, args, dev_args, 1, use_optional)
        h = run_host(mpc, host_name, args, use_optional, lane)
        assert sorted(h) == sorted(d0), host_name
        for k in h:
            a, what = args[k], f"{host_name} arg {k} optional={use_optional}"
            hb, b0, b1 = bits(h[k]).ravel(), bits(d0[k]).ravel(), bits(d1[k]).ravel()
            if a.kind == "out":
                # elements the kernel leaves alone hold whatever the staging held: compare what the device form writes
                s0, s1 = bits(np.array([SENTINELS[a.dtype][0]], a.dtype))[0], bits(np.array([SENTINELS[a.dtype][1]], a.dtype))[0]
                b0, b1 = b0[:hb.size], b1[:hb.size]
                written = ~((b0 == s0) & (b1 == s1))
                assert np.array_equal(b0[written], b1[written]), what + ": device form not deterministic"
                assert np.array_equal(hb[written], b0[written]), what
            else:
                assert np.array_equal(hb, b0), what


def with_stream(p):
    return p + [None]


# ---------------------------------------------------------------------------------------------- entry specs
def spec_qp(mpc, B, seed):
    n, p, m = 6, 1, 8
    d = synth.random_qp(B, n, p, m, seed=seed)
    args = [n, p, m, B, Buf("in", d["G"]), Buf("in", d["g0"]), Buf("in", d["CE"]), Buf("in", d["ce0"]), Buf("in", d["CI"]),
            Buf("in", d["ci0"]), Buf("inout", np.zeros((B, n))), Buf("out", shape=(B,), optional=True),
            Buf("out", shape=(B * (m + p),), dtype=np.int32, optional=True, dev_shape=(B * (m + p + 1),)),
            Buf("out", shape=(B,), dtype=np.int32, optional=True), Buf("out", shape=(B, 6), dtype=np.int32, optional=True),
            Buf("out", shape=(B,), dtype=np.int32, optional=True)]
    return "go1mpc_qp_solve_batch_host", "go1mpc_qp_solve_batch", args, with_stream


def body_record(B, seed):
    d = synth.body_mpc_inputs(B, NH, seed=seed)
    rec = q.pack_body_inputs(NH, d["tick"], d["tx"], d["theta"], d["bstate"], d["x_warm"], d["refs"])
    out = np.zeros((B, q.body_out_stride(NH)))
    out[:, 18:18 + 2 * NH] = d["x_warm"]
    return rec, out


def spec_body(mpc, B, seed):
    rec, out = body_record(B, seed)
    args = [NH, B, Buf("in", rec), Buf("inout", out), Buf("out", shape=(B, q.body_diag_stride(NH)), dtype=np.int32, optional=True)]
    return "go1mpc_body_mpc_step_batch_host", "go1mpc_body_mpc_step_batch", args, with_stream


def step_inputs(mpc, B, seed):
    tick, st, sin = synth.step_timing_inputs(B, mpc.step_default_state(), seed=seed)
    return np.ascontiguousarray(tick, np.int32), soa(st), soa(sin)


def spec_step(mpc, B, seed):
    tick, st, sin = step_inputs(mpc, B, seed)
    args = [3, B, Buf("in", tick), Buf("inout", st), Buf("in", sin), Buf("out", shape=(q.STEP_OUT, B)),
            Buf("out", shape=(q.STEP_DIAG, B), dtype=np.int32, optional=True)]
    return ("go1mpc_step_timing_step_batch_host", "go1mpc_step_timing_step_batch", args,
            lambda p: p[:4] + [p[3]] + p[4:] + [None])     # in place: state_out = state


def foot_inputs(mpc, B, seed):
    """A planner tick's real results, so that the swing-foot kernel sees consistent step tables."""
    tick, st, sin = step_inputs(mpc, B, seed)
    host = spec_step(mpc, B, seed)
    out38 = cleared(run_device(mpc, host[0], host[1], host[2], host[3], 0, True)[5])
    return tick, st, out38, soa(np.tile(mpc.foot_default_state(), (B, 1)))


def spec_foot(mpc, B, seed):
    tick, st, out38, foot = foot_inputs(mpc, B, seed)
    args = [B, Buf("in", tick), Buf("in", st), Buf("in", out38), Buf("inout", foot), Buf("out", shape=(18, B)),
            Buf("out", shape=(B,), dtype=np.int32, optional=True)]
    return "go1mpc_foot_trajectory_batch_host", "go1mpc_foot_trajectory_batch", args, with_stream


def spec_foot_stop(mpc, B, seed):
    tick, st, out38, foot = foot_inputs(mpc, B, seed)
    lift0 = np.full(B, 27.0)            # the planner node's initial value (GO1MPC_FOOTSTEPS)
    stop = (np.arange(B) % 3 == 0).astype(np.float64)
    args = [B, Buf("in", tick), Buf("in", st), Buf("in", out38), Buf("inout", foot), Buf("out", shape=(18, B)),
            Buf("out", shape=(B,), dtype=np.int32, optional=True), Buf("inout", lift0), Buf("in", stop, optional=True)]
    return "go1mpc_foot_trajectory_stop_batch_host", "go1mpc_foot_trajectory_stop_batch", args, with_stream


def spec_grf_opt(mpc, B, seed):
    d = grf_inputs(B, seed=seed)
    rec = np.zeros((B, 48))
    rec[:, 0:3] = d["base"]; rec[:, 3:15] = d["legs"]; rec[:, 15:21] = d["FT"]; rec[:, 21:33] = d["prev"]; rec[:, 33:45] = d["prev"]
    rec[:, 45] = d["mode"]; rec[:, 46] = d["rs"]
    args = [B, Buf("in", rec), Buf("out", shape=(B, 16)), Buf("out", shape=(B, 32), dtype=np.int32, optional=True)]
    return "go1mpc_grf_force_opt_batch_host", "go1mpc_grf_force_opt_batch", args, with_stream


def spec_grf_dist(mpc, B, seed):
    d = grf_inputs(B, seed=seed)
    args = [B, 102, 0.9] + [Buf("in", soa(d[k])) for k in ("base", "legs", "F6", "rf", "lf")] + [Buf("out", shape=(12, B))]
    return "go1mpc_grf_force_distribution_batch_host", "go1mpc_grf_force_distribution_batch", args, with_stream


def spec_grf_tau(mpc, B, seed):
    d = tau_inputs(B, seed=seed)
    args = ([B] + [Buf("in", soa(d[k])) for k in ("jac", "swing", "p_des", "p_est", "pv_des", "pv_est", "F")] +
            [B, 1, Buf("out", shape=(12, B))])
    return "go1mpc_grf_joint_torques_batch_host", "go1mpc_grf_joint_torques_batch", args, with_stream


def nlp_inputs(mpc, B, seed):
    rng = np.random.default_rng(seed)
    st = soa(np.tile(mpc.nlp_node_default_state(), (B, 1)))
    wd = (np.arange(B) % 40 + 1).astype(np.int32)
    start = np.ones(B, np.int32)
    cmd = np.zeros(B, np.int32)
    rf = rng.uniform(-0.01, 0.01, (3, B)); lf = rng.uniform(-0.01, 0.01, (3, B))
    return st, wd, start, cmd, rf, lf


def spec_nlp(mpc, B, seed):
    st, wd, start, cmd, rf, lf = nlp_inputs(mpc, B, seed)
    args = [B, Buf("inout", st), Buf("in", wd), Buf("in", start, optional=True), Buf("in", cmd, optional=True),
            Buf("in", rf, optional=True), Buf("in", lf, optional=True), Buf("out", shape=(100, B))]
    return "go1mpc_nlp_node_tick_batch_host", "go1mpc_nlp_node_tick_batch", args, with_stream


def spec_rt(mpc, B, seed):
    import torch
    nlp = spec_nlp(mpc, B, seed)
    msg = cleared(run_device(mpc, nlp[0], nlp[1], nlp[2], nlp[3], 0, True)[7])      # a planner message the node consumes
    st = soa(np.tile(mpc.rt_node_default_state(NH), (B, 1)))
    body_in = torch.zeros(B, q.body_in_stride(NH), dtype=torch.float64, device="cuda")
    args = [NH, B, Buf("inout", st), Buf("in", msg), Buf("in", np.zeros(B, np.int32), optional=True),
            Buf("in", np.zeros((4, B)), optional=True), Buf("inout", np.zeros((B, q.body_out_stride(NH)))), Buf("out", shape=(100, B))]
    # device form: the body-MPC input records are a caller buffer; no body diagnostics, every robot active
    return ("go1mpc_rt_node_tick_batch_host", "go1mpc_rt_node_tick_batch", args,
            lambda p: p[:6] + [body_in.data_ptr(), p[6], None, p[7], None, None])


def leg_inputs(B, seed):
    rng = np.random.default_rng(seed)
    qj = soa(np.array([0.0, 0.7, -1.4]) + rng.uniform(-0.2, 0.2, (B, 3)))
    leg = (np.arange(B) % 4).astype(np.int32)
    return qj, leg, rng.uniform(-0.02, 0.02, (3, B)), rng.uniform(-0.1, 0.1, (3, B))


def spec_leg_fk(mpc, B, seed):
    qj, leg, bp, br = leg_inputs(B, seed)
    args = [B, Buf("in", qj), Buf("in", leg), Buf("in", bp, optional=True), Buf("in", br, optional=True), Buf("out", shape=(3, B)),
            Buf("out", shape=(9, B), optional=True)]
    return "go1mpc_leg_fk_batch_host", "go1mpc_leg_fk_batch", args, with_stream


def spec_leg_ik(mpc, B, seed):
    qj, leg, bp, br = leg_inputs(B, seed)
    fk = spec_leg_fk(mpc, B, seed)
    pdes = cleared(run_device(mpc, fk[0], fk[1], fk[2], fk[3], 0, False)[5])
    args = [B, Buf("in", pdes), Buf("in", qj + 0.05), Buf("in", leg), Buf("in", bp, optional=True), Buf("in", br, optional=True),
            Buf("out", shape=(3, B)), Buf("out", shape=(9, B), optional=True), Buf("out", shape=(B,), dtype=np.int32, optional=True)]
    return "go1mpc_leg_ik_batch_host", "go1mpc_leg_ik_batch", args, with_stream


SYNC_SPECS = [spec_qp, spec_body, spec_step, spec_foot, spec_foot_stop, spec_grf_opt, spec_grf_dist, spec_grf_tau, spec_nlp, spec_rt,
              spec_leg_fk, spec_leg_ik]


def test_sync_host_entries_equal_device_forms():
    """Each synchronous host entry equals its device form bit for bit at every size, optional buffers given or NULL."""
    mpc = q.Go1Mpc()
    try:
        for i, B in enumerate(SIZES):
            for spec in SYNC_SPECS:
                check_entry(mpc, spec(mpc, B, 100 + 10 * i + B % 7))
    finally:
        mpc.close()


# ---------------------------------------------------------------------------------------------- lane entries
def spec_body_lane(mpc, B, seed):
    rec, _ = body_record(B, seed)        # ticks 100..1700: none is gated, so the lane does not upload the previous out records
    args = [NH, B, Buf("in", rec), Buf("out", shape=(B, q.body_out_stride(NH))),
            Buf("out", shape=(B, q.body_diag_stride(NH)), dtype=np.int32, optional=True)]
    return "go1mpc_body_mpc_step_batch_host_async", "go1mpc_body_mpc_step_batch", args, with_stream


def spec_step_lane(mpc, B, seed):
    tick, st, sin = step_inputs(mpc, B, seed)
    args = [3, B, Buf("in", tick), Buf("dev", st), Buf("dev", st + 0.0), Buf("in", sin), Buf("out", shape=(q.STEP_OUT, B)),
            Buf("out", shape=(q.STEP_DIAG, B), dtype=np.int32, optional=True)]
    return "go1mpc_step_timing_step_batch_host_async", "go1mpc_step_timing_step_batch", args, with_stream


def check_resident_lane(mpc, B, seed, with_diag):
    """The resident-record lane against the device form on the full records it expands."""
    import torch
    d = synth.body_mpc_inputs(B, NH, seed=seed)
    rec, out = body_record(B, seed)
    tx, _, tick = q.split_body_record(NH, rec)
    ds = q.body_diag_stride(NH)
    want_out = torch.from_numpy(out.copy()).cuda()
    want_diag = torch.zeros(B, ds, dtype=torch.int32, device="cuda")
    full = q.pack_body_inputs(NH, d["tick"], d["tx"], d["theta"], d["bstate"], out[:, 18:18 + 2 * NH], d["refs"])
    mpc.body_mpc_step(NH, B, torch.from_numpy(full).cuda(), want_out, want_diag)
    mpc.synchronize()
    tx_d, out_d = torch.from_numpy(tx).cuda(), torch.from_numpy(out.copy()).cuda()
    t_out = np.full((B, q.BODY_TICK_OUT), np.nan)
    diag = np.full((B, ds), -7, np.int32) if with_diag else None
    torch.cuda.synchronize()
    mpc.body_mpc_step_resident_host_async(NH, B, tx_d, out_d, np.ascontiguousarray(tick), t_out, diag)
    mpc.synchronize()
    o = want_out.cpu().numpy()
    assert np.array_equal(bits(out_d.cpu().numpy()), bits(o))
    assert np.array_equal(bits(t_out[:, :18]), bits(o[:, :18]))
    assert np.array_equal(bits(t_out[:, 18]), bits(o[:, 18 + 2 * NH]))
    if with_diag:
        assert np.array_equal(diag, want_diag.cpu().numpy())


def test_lane_entries_equal_device_forms():
    """The three pipelined host entries, after go1mpc_synchronize, equal the device forms bit for bit."""
    mpc = q.Go1Mpc()
    try:
        for i, B in enumerate(SIZES):
            seed = 500 + 10 * i + B % 7
            check_entry(mpc, spec_body_lane(mpc, B, seed), lane=True)
            check_entry(mpc, spec_step_lane(mpc, B, seed), lane=True)
            for with_diag in (True, False):
                check_resident_lane(mpc, B, seed, with_diag)
    finally:
        mpc.close()


# ---------------------------------------------------------------------------------------------- stream limit
def test_stream_limit_is_one_count_per_handle():
    """256 distinct streams work; the 257th is refused with GO1MPC_E_UNSUPPORTED before anything is enqueued."""
    import torch
    torch.cuda.init()
    torch.zeros(1, device="cuda")          # the primary context is current on this thread
    cu = ctypes.CDLL("libcuda.so.1")
    mpc = q.Go1Mpc()
    streams = []
    try:
        B = 4
        rec, out = body_record(B, 9)
        rec_d = torch.from_numpy(rec).cuda()
        for k in range(257):
            s = ctypes.c_void_p()
            assert cu.cuStreamCreate(ctypes.byref(s), 1) == 0
            streams.append(s)
        out_d = torch.from_numpy(out).cuda()
        torch.cuda.synchronize()
        for k in range(256):
            rc = mpc.lib.go1mpc_body_mpc_step_batch(mpc.h, NH, B, rec_d.data_ptr(), out_d.data_ptr(), None, streams[k])
            assert rc == 0, (k, mpc.lib.go1mpc_last_error(mpc.h).decode())
            cu.cuStreamSynchronize(streams[k])
        fresh = torch.full_like(out_d, 3.25)
        n0 = mpc.launch_count
        torch.cuda.synchronize()
        rc = mpc.lib.go1mpc_body_mpc_step_batch(mpc.h, NH, B, rec_d.data_ptr(), fresh.data_ptr(), None, streams[256])
        assert rc == -4, rc
        assert "256" in mpc.lib.go1mpc_last_error(mpc.h).decode()
        assert mpc.launch_count == n0
        cu.cuStreamSynchronize(streams[256])
        assert (fresh == 3.25).all()
        # a stream already known keeps working
        rc = mpc.lib.go1mpc_body_mpc_step_batch(mpc.h, NH, B, rec_d.data_ptr(), fresh.data_ptr(), None, streams[0])
        assert rc == 0
        cu.cuStreamSynchronize(streams[0])
    finally:
        mpc.close()
        for s in streams:
            cu.cuStreamDestroy_v2(s)
