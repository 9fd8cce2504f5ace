"""Episode farm on a GPU: per-robot clocks and on-device resets of the gait stack, one JSON line per run.

Setup: B in --batch (default 4096, 65536), nh = 10, sensor rows from 16 seeded pinned buffers (gait_stack_probe.sensors), result
rows copied to a pinned host buffer on every call.  Each mode gets its own batch, walked --warm periods into the gait first, then
the device time (CUDA events on the handle's stream) of --reps windows of 10 consecutive 10 ms periods -- two planner cycles, no
host synchronisation inside a window -- is divided by 10:
  a_host_schedule    go1mpc_gait_stack_tick_host_async, planner flag from the reference's schedule (4 planner periods in 10)
  b_clocked_aligned  go1mpc_gait_stack_tick_clocked_async, every clock started together (the same 4 planner periods in 10)
  c_clocked_spread   the clocked entry with the robots' clocks spread uniformly over c mod 5 (staggered by resets in the first five
                     warm-up periods): every period about 40 % of the robots plan, and the planner kernels run every period
  d_spread_resets    (c) plus 1 % of the robots reset every period, the reset call included
  e_graph_period     one captured period -- reset (1 % flagged) + clocked tick + servo stack K = 10 -- replayed; e_direct_period is
                     the same period enqueued call by call, for the launch overhead the graph removes
Reported per mode: median, p10 and p90 of the per-period mean over the windows.  gpu: name, power limit and SM clock, read in the
same run before and after.
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

NH, K, WINDOW = 10, 10, 10
Q0 = np.tile(ssp.QH, 4)


class EpisodeFarm:
    """B robots on the clocked entry with pinned host buffers; optional resets and servo calls per period."""

    def __init__(self, mpc, B, seed, servo=False, n_sensors=16):
        import torch
        import quadrupedal_loco_b200 as q
        self.mpc, self.B = mpc, B
        col = mpc.gait_stack_default_state(NH)
        self.state = torch.from_numpy(np.repeat(col[:, None], B, axis=1).copy()).cuda()
        self.body_out = torch.zeros(B, q.body_out_stride(NH), dtype=torch.float64, device="cuda")
        self.rows_d = torch.zeros(B, len(gsp.SLOTS), dtype=torch.float64, device="cuda")
        self.rows = torch.zeros(B, len(gsp.SLOTS), dtype=torch.float64).pin_memory()
        self.clock = torch.zeros(B, dtype=torch.int32, device="cuda")
        self.servo = ssp.servo_state(mpc, B) if servo else None
        self.q_d = torch.zeros(B, 12 * K, dtype=torch.float64, device="cuda")
        self.sens = [torch.from_numpy(s).pin_memory() for s in gsp.sensors(B, n_sensors, seed)]
        self.t = [mpc.gait_stack_tick_clocked_struct(NH, s, self.clock, self.state, self.body_out, gsp.SLOTS, self.rows_d, self.rows)
                  for s in self.sens]
        b = np.arange(B)
        # resets: staggering (robots with b mod 5 = i in warm-up period i), and 1 % of the robots per period (b mod 100 = i)
        self.stagger = [self._flags(b % 5 == i) for i in range(5)]
        self.churn = [self._flags(b % 100 == i) for i in range(WINDOW)]
        self.k = 0
        torch.cuda.synchronize()

    def _flags(self, mask):
        import torch
        fl = torch.from_numpy(mask.astype(np.int32)).pin_memory()
        return fl, self.mpc.gait_stack_reset_struct(NH, fl, self.clock, self.state, self.body_out, self.servo, Q0)

    def call(self, reset=None):
        if reset is not None:
            self.mpc.gait_stack_reset_async(self.B, reset[1])
        self.mpc.gait_stack_tick_clocked_async(self.B, self.t[self.k % len(self.sens)])
        if self.servo is not None:
            self.mpc.servo_stack_tick(self.B, K, 102, 1.0, self.state, self.servo, self.q_d)
        self.k += 1


def windows(mpc, reps, period):
    """Per-period device time (us) of `reps` windows of WINDOW consecutive periods."""
    import torch
    s = torch.cuda.ExternalStream(mpc.stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(reps):
        mpc.synchronize()
        e0.record(s)
        for i in range(WINDOW):
            period(i)
        e1.record(s); e1.synchronize()
        out.append(e0.elapsed_time(e1) * 1e3 / WINDOW)
    return out


def stats(v):
    return {"median": float(np.median(v)), "p10": float(np.percentile(v, 10)), "p90": float(np.percentile(v, 90))}


def measure(mpc, B, warm, reps):
    import torch
    res = {"B": B, "nh": NH, "warm_periods": warm, "reps": reps, "periods_per_window": WINDOW}
    # (a) the existing entry on the host schedule
    f = gsp.Farm(mpc, NH, B, seed=1000 + B)
    for _ in range(warm):
        f.call()
    res["a_host_schedule"] = stats(windows(mpc, reps, lambda i: f.call()))
    del f
    # (b) clocked, aligned
    f = EpisodeFarm(mpc, B, seed=1000 + B)
    for _ in range(warm):
        f.call()
    res["b_clocked_aligned"] = stats(windows(mpc, reps, lambda i: f.call()))
    del f
    # (c) clocked, spread over c mod 5;  (d) the same plus 1 % resets per period
    f = EpisodeFarm(mpc, B, seed=1000 + B)
    for p in range(warm):
        f.call(f.stagger[p] if p < 5 else None)
    c = f.clock.cpu().numpy()
    res["clock_residues_c"] = np.bincount(c % 5, minlength=5).tolist()
    res["c_clocked_spread"] = stats(windows(mpc, reps, lambda i: f.call()))
    res["d_spread_resets"] = stats(windows(mpc, reps, lambda i: f.call(f.churn[i])))
    del f
    # (e) one captured period: reset (1 %) + clocked tick + servo K = 10, against the same period enqueued directly
    f = EpisodeFarm(mpc, B, seed=1000 + B, servo=True)
    for p in range(warm):
        f.call(f.stagger[p] if p < 5 else None)
    res["e_direct_period"] = stats(windows(mpc, reps, lambda i: f.call(f.churn[0])))
    mpc.synchronize()
    st = mpc.stream
    mpc._check(mpc.lib.go1mpc_graph_capture_begin(mpc.h, st), "capture_begin")
    f.call(f.churn[0])
    ge = ctypes.c_void_p()
    mpc._check(mpc.lib.go1mpc_graph_capture_end(mpc.h, st, ctypes.byref(ge)), "capture_end")
    try:
        for _ in range(3):
            mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, st), "graph_launch")
        res["e_graph_period"] = stats(windows(mpc, reps, lambda i: mpc._check(mpc.lib.go1mpc_graph_launch(mpc.h, ge, st), "graph_launch")))
    finally:
        mpc.synchronize()
        mpc._check(mpc.lib.go1mpc_graph_destroy(mpc.h, ge), "graph_destroy")
    del f
    torch.cuda.empty_cache()
    res["c_over_a"] = res["c_clocked_spread"]["median"] / res["a_host_schedule"]["median"]
    res["b_over_a"] = res["b_clocked_aligned"]["median"] / res["a_host_schedule"]["median"]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--warm", type=int, default=200, help="periods walked before timing")
    ap.add_argument("--reps", type=int, default=30, help="timed windows of 10 periods per mode")
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
