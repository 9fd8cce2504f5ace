"""Farm column copy (go1mpc_farm_copy_async) on a GPU: one JSON line per run.

Setup: a farm of B robots (default 65536), nh = 10, with every block a copy can carry -- gait stack state, body records, clocks,
servo state, force state -- walked --warm periods into the gait (clocked tick + K = 10 torque tick, clocks staggered over c mod 5
by resets in the first five periods).  At nh = 10 a robot is 11 636 B, so the farm is larger than the 126 MB L2 and every full
copy streams through HBM.  Device time of each mode on the handle's stream (CUDA events, median / p10 / p90 over --reps calls,
the modes alternated within each rep, after warm-up calls of each):
  a_restore_all      every robot restored from a 64-column bank (index i -> i mod 64)
  b_restore_1pct     1 % of the robots restored from the bank, -1 elsewhere
  c_snapshot_ident   every robot snapshotted into a full-size bank, identity index
  d_snapshot_perm    the same with a random permutation as index
  e_fork_one         one bank column forked into every robot
  memcpy_farm        cudaMemcpyAsync device-to-device of the farm's five blocks into the full-size bank (go1mpc_copy_device_async):
                     the reference for (a) to (e), same bytes, same process
  f_period / f_period_restore  one captured period (clocked tick + torque tick K = 10) replayed, without and with a 1 % restore
                     in front
Bytes written per second = copied robots x robot bytes / time.  gpu: name, power limit and SM clock, read in the same run before and
after.
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.append(os.path.dirname(HERE))
sys.path.append(HERE)
import gait_stack_probe as gsp  # noqa: E402
import servo_stack_probe as ssp  # noqa: E402

NH, K, GM, BANK = 10, 10, 102, 64
Q0 = np.tile(ssp.QH, 4)


class Robots:
    """One farm-shaped buffer set; with sensors, the clocked tick and torque tick run on it."""

    def __init__(self, mpc, B, seed=None):
        import torch
        import quadrupedal_loco_b200 as q
        f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device="cuda")
        self.mpc, self.B = mpc, B
        col = mpc.gait_stack_default_state(NH)
        self.state = torch.from_numpy(np.repeat(col[:, None], B, axis=1).copy()).cuda()
        self.body_out = f64(B, q.body_out_stride(NH))
        self.clock = torch.zeros(B, dtype=torch.int32, device="cuda")
        self.servo = ssp.servo_state(mpc, B)
        self.force = f64(q.SERVO_FORCE_ROWS, B)
        self.cols = mpc.farm_columns(B, self.state, self.body_out, self.clock, self.servo, self.force)
        if seed is None:
            return
        rng = np.random.Generator(np.random.Philox(seed))
        self.meas = torch.from_numpy(np.concatenate([Q0[:, None] + rng.uniform(-0.1, 0.1, (12, B)), rng.uniform(-3, 3, (12, B))])).cuda()
        self.rows_d, self.q_d, self.tau_d = f64(B, len(gsp.SLOTS)), f64(B, 12 * K), f64(B, 12 * K)
        self.sens = [torch.from_numpy(s).pin_memory() for s in gsp.sensors(B, 16, seed)]
        self.t = [mpc.gait_stack_tick_clocked_struct(NH, s, self.clock, self.state, self.body_out, gsp.SLOTS, self.rows_d) for s in self.sens]
        self.k = 0

    def period(self):
        self.mpc.gait_stack_tick_clocked_async(self.B, self.t[self.k % len(self.sens)])
        self.mpc.servo_torque_tick(self.B, K, GM, 1.0, 0.9, self.state, self.servo, self.force, self.meas, self.q_d, self.tau_d)
        self.k += 1

    def blocks(self):
        return (self.state, self.body_out, self.clock, self.servo, self.force)


def stats(v):
    return {"median": float(np.median(v)), "p10": float(np.percentile(v, 10)), "p90": float(np.percentile(v, 90))}


def measure(mpc, B, warm, reps):
    import torch
    import quadrupedal_loco_b200 as q
    robot_bytes = 8 * (mpc.gait_stack_state_doubles(NH) + q.body_out_stride(NH) + q.SERVO_STATE_ROWS + q.SERVO_FORCE_ROWS) + 4
    farm = Robots(mpc, B, seed=3000 + B)
    bank = Robots(mpc, BANK)
    full = Robots(mpc, B)
    b = np.arange(B)
    rng = np.random.default_rng(B)
    stagger = [torch.from_numpy((b % 5 == i).astype(np.int32)).pin_memory() for i in range(5)]
    torch.cuda.synchronize()
    for p in range(warm):
        if p < 5:
            mpc.gait_stack_reset_async(B, mpc.gait_stack_reset_struct(NH, stagger[p], farm.clock, farm.state, farm.body_out, farm.servo, Q0))
        farm.period()
    ix = lambda a: torch.as_tensor(np.asarray(a, dtype=np.int32), device="cuda")
    sel = rng.choice(B, B // 100, replace=False)
    one_pct = np.full(B, -1); one_pct[sel] = sel % BANK
    index = {"a_restore_all": ix(b % BANK), "b_restore_1pct": ix(one_pct), "c_snapshot_ident": ix(b),
             "d_snapshot_perm": ix(rng.permutation(B)), "e_fork_one": ix(np.zeros(B))}
    copied = {"a_restore_all": B, "b_restore_1pct": len(sel), "c_snapshot_ident": B, "d_snapshot_perm": B, "e_fork_one": B}
    torch.cuda.synchronize()
    mpc.farm_copy(NH, bank.cols, farm.cols, ix(b[:BANK] * (B // BANK)))      # a bank of 64 walking robots
    farm_cols, bank_cols, full_cols = farm.cols, bank.cols, full.cols

    def memcpy():
        for d, s in zip(full.blocks(), farm.blocks()):
            mpc._check(mpc.lib.go1mpc_copy_device_async(mpc.h, d.data_ptr(), s.data_ptr(), d.numel() * d.element_size(), None), "copy")

    modes = {
        "a_restore_all": lambda: mpc.farm_copy(NH, farm_cols, bank_cols, index["a_restore_all"]),
        "b_restore_1pct": lambda: mpc.farm_copy(NH, farm_cols, bank_cols, index["b_restore_1pct"]),
        "c_snapshot_ident": lambda: mpc.farm_copy(NH, full_cols, farm_cols, index["c_snapshot_ident"]),
        "d_snapshot_perm": lambda: mpc.farm_copy(NH, full_cols, farm_cols, index["d_snapshot_perm"]),
        "e_fork_one": lambda: mpc.farm_copy(NH, farm_cols, bank_cols, index["e_fork_one"]),
        "memcpy_farm": memcpy,
    }
    s = torch.cuda.ExternalStream(mpc.stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t = {m: [] for m in modes}
    for fn in modes.values():
        for _ in range(3):
            fn()
    mpc.synchronize()
    for _ in range(reps):
        for m, fn in modes.items():
            e0.record(s); fn(); e1.record(s); e1.synchronize()
            t[m].append(e0.elapsed_time(e1) * 1e3)
    res = {"B": B, "nh": NH, "robot_bytes": robot_bytes, "farm_bytes": robot_bytes * B, "bank_columns": BANK, "warm_periods": warm,
           "reps": reps}
    for m, v in t.items():
        n = copied.get(m, B)
        res[m] = dict(us=stats(v), robots=n, gb_written_per_s=n * robot_bytes / (np.median(v) * 1e-6) / 1e9)
    mc = np.median(t["memcpy_farm"])
    for m in ("a_restore_all", "c_snapshot_ident", "d_snapshot_perm", "e_fork_one"):
        res[m]["over_memcpy"] = float(np.median(t[m]) / mc)
    res["target_1p5x_met"] = bool(res["a_restore_all"]["over_memcpy"] <= 1.5 and res["c_snapshot_ident"]["over_memcpy"] <= 1.5)

    # (f) one captured period, without and with a 1 % restore in front (the index stays fixed: the work is the same every period)
    st = mpc.stream

    def capture(fn):
        mpc.synchronize()
        mpc._check(mpc.lib.go1mpc_graph_capture_begin(mpc.h, st), "capture_begin")
        fn()
        ge = ctypes.c_void_p()
        mpc._check(mpc.lib.go1mpc_graph_capture_end(mpc.h, st, ctypes.byref(ge)), "capture_end")
        return ge

    def with_restore():
        mpc.farm_copy(NH, farm_cols, bank_cols, index["b_restore_1pct"])
        farm.period()

    graphs = {"f_period": capture(farm.period), "f_period_restore": capture(with_restore)}
    tf = {m: [] for m in graphs}
    try:
        for ge in graphs.values():
            for _ in range(3):
                mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, st), "graph_launch")
        mpc.synchronize()
        for _ in range(reps):
            for m, ge in graphs.items():
                e0.record(s)
                mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, st), "graph_launch")
                e1.record(s); e1.synchronize()
                tf[m].append(e0.elapsed_time(e1) * 1e3)
    finally:
        mpc.synchronize()
        for ge in graphs.values():
            mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
    for m, v in tf.items():
        res[m] = {"us": stats(v)}
    res["clock_residues"] = np.bincount(farm.clock.cpu().numpy() % 5, minlength=5).tolist()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, nargs="+", default=[65536])
    ap.add_argument("--warm", type=int, default=40, help="periods walked before timing")
    ap.add_argument("--reps", type=int, default=30, help="timed calls per mode")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import quadrupedal_loco_b200 as q
    mpc = q.Go1Mpc(0)
    res = {"gpu": gsp.gpu_info(), "runs": [measure(mpc, B, a.warm, a.reps) for B in a.batch], "gpu_after": gsp.gpu_info()}
    mpc.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
