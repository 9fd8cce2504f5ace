"""Servo torque tick (go1mpc_servo_torque_tick_async) on a GPU: one JSON line per run.

Setup: B in --batch (default 4096, 65536), nh = 10, every robot walked --warm periods into the gait on the reference's clock
(gait stack call + K = 10 torque call per 10 ms period), then in the same process:
  torque_us   (a) device time (CUDA events, median over --reps) of one K = 10 torque call
  chained_us  (b) the same period from the single-stage entries: one K = 10 servo stack call + 10 x (force distribution, force QP,
              joint torques) = 30 GRF launches, timed alternately with (a).  The records those launches read are assembled once
              outside the timed window, so (b) leaves out the glue kernels a caller needs between them: a lower bound
  period      (c) sustained 10 ms periods per second of gait stack call + K = 10 torque call with q and tau copied to pinned
              host buffers, over at least --window s; the share of a 10 ms period one takes
  bytes_per_robot_period  PCIe bytes of a period, counted from the layouts
  gpu         name, power limit and SM clock, read in the same run
"""
import argparse
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.append(os.path.dirname(HERE))
sys.path.append(HERE)
import gait_stack_probe as gsp  # noqa: E402
from servo_stack_probe import servo_state  # noqa: E402

K = 10
GM = 102


def measure(mpc, B, warm, reps, window):
    import torch
    import quadrupedal_loco_b200 as q
    f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device="cuda")
    f = gsp.Farm(mpc, 10, B, seed=2000 + B)
    sv = servo_state(mpc, B)
    rng = np.random.Generator(np.random.Philox(B))
    meas = torch.from_numpy(np.concatenate([np.tile([0, 0.87, -1.5], 4)[:, None] + rng.uniform(-0.1, 0.1, (12, B)),
                                            rng.uniform(-3, 3, (12, B))])).cuda()
    force, q_d, tau_d = f64(q.SERVO_FORCE_ROWS, B), f64(B, 12 * K), f64(B, 12 * K)
    q_h = torch.zeros(B, 12 * K, dtype=torch.float64).pin_memory(); t_h = torch.zeros_like(q_h).pin_memory()

    def torque(host=False):
        mpc.servo_torque_tick(B, K, GM, 1.0, 0.9, f.state, sv, force, meas, q_d, tau_d, **(dict(q=q_h, tau=t_h) if host else {}))

    for _ in range(warm):
        f.call()
        torque()
    mpc.synchronize()
    s = torch.cuda.ExternalStream(mpc.stream)
    # (b): records of one tick, built once (the chained launches then run on fixed inputs)
    sv_c, jac, fd = sv.clone(), f64(36, B), f64(12, B)
    gait = f.state[q.STACK_ROW_GAIT:q.STACK_ROW_GAIT + 100]
    com, fref, rec, out, diag = f64(3, B), f64(12, B), f64(B, 48), f64(B, 16), torch.zeros(B, 32, dtype=torch.int32, device="cuda")
    swing = torch.zeros(4, B, dtype=torch.int32, device="cuda")
    pest, pvdes, pvest, tau = f64(12, B), f64(12, B), f64(12, B), f64(12, B)
    q10 = f64(B, 12 * K)
    with torch.cuda.stream(s):
        mpc.servo_stack_tick(B, 1, GM, 1.0, f.state, sv_c, q10[:, :12].contiguous(), jac_d=jac, foot_des_d=fd)
        ch = sv_c[q.SERVO_ROW_LPF + 27:q.SERVO_ROW_LPF + 36]
        com.copy_(torch.stack([ch[0], ch[1], ch[2]]))
        rec[:, 0:3] = com.T; rec[:, 3:15] = fd.T; rec[:, 45] = GM; rec[:, 46] = gait[99]
        F6, rf, lf = gait[15:21].contiguous(), ch[6:9].contiguous(), ch[3:6].contiguous()
    torch.cuda.synchronize()

    def chained():
        mpc.servo_stack_tick(B, K, GM, 1.0, f.state, sv_c, q10)
        for _ in range(K):
            mpc.grf_force_distribution(B, GM, 0.9, com, fd, F6, rf, lf, fref)
            mpc.grf_force_opt(B, rec, out, diag)
            mpc.grf_joint_torques(B, jac, swing, fd, pest, pvdes, pvest, out, tau, F_strides=(1, 16))

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    t = {"torque": [], "chained": []}
    for _ in range(3):
        torque(); chained()
    mpc.synchronize()
    for _ in range(reps):
        for name, fn in (("torque", torque), ("chained", chained)):
            ev[0].record(s); fn(); ev[1].record(s); ev[1].synchronize()
            t[name].append(ev[0].elapsed_time(ev[1]) * 1e3)
    n = 0
    t0 = time.perf_counter()
    while True:
        for _ in range(10):
            f.call()
            torque(host=True)
            n += 1
        mpc.synchronize()
        el = time.perf_counter() - t0
        if el >= window:
            break
    stat = lambda v: {"median": float(np.median(v)), "p10": float(np.percentile(v, 10)), "p90": float(np.percentile(v, 90))}
    return {
        "B": B, "nh": 10, "K": K, "gait_mode": GM, "warm_periods": warm, "reps": reps,
        "torque_us": stat(t["torque"]), "chained_us": stat(t["chained"]),
        "speedup": float(np.median(t["chained"]) / np.median(t["torque"])),
        "period": {"seconds": el, "periods": n, "periods_per_s": n / el, "robot_periods_per_s": B * n / el,
                   "share_of_10ms": el / n / 0.010},
        "bytes_per_robot_period": {"h2d_sensor": gsp.SENSOR_ROWS * 8, "h2d_meas_when_copied": 24 * 8, "d2h_q": 12 * K * 8,
                                   "d2h_tau": 12 * K * 8, "d2h_stack_rows": len(gsp.SLOTS) * 8},
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--warm", type=int, default=200, help="periods walked before timing")
    ap.add_argument("--reps", type=int, default=50, help="timed calls per mode")
    ap.add_argument("--window", type=float, default=1.0, help="seconds of back-to-back periods (>= 0.2)")
    a = ap.parse_args()
    assert a.window >= 0.2
    import quadrupedal_loco_b200 as q
    mpc = q.Go1Mpc(0)
    res = {"gpu": gsp.gpu_info(), "runs": [measure(mpc, B, a.warm, a.reps, a.window) for B in a.batch], "gpu_after": gsp.gpu_info()}
    mpc.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
