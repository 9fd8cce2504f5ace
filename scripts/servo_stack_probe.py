"""Servo stack tick (go1mpc_servo_stack_tick_async) on a GPU: one JSON line per run.

Setup: B in --batch (default 4096, 65536), nh = 10, every robot walked --warm fast ticks into the gait on the reference's clock
(planner every 25 ms, fast node every 10 ms) with a K = 10 servo call after each gait stack call, as gait_stack_probe.py does,
then in the same process:
  fused_us / chained_us  device time (CUDA events, median over --reps) of one K = 10 servo call and of the same ten ticks as
                         10 x (go1mpc_lpf_batch + go1mpc_servo_kin_tick_batch), measured alternately on copies of one servo state
                         (the chained theta rows are gathered outside the timed window)
  period                 sustained 10 ms periods per second of gait stack call + K = 10 servo call with the joint targets copied
                         to a pinned host buffer, over at least --window s; the share of a 10 ms period one takes
  bytes_per_robot_period PCIe bytes of a period (sensor rows up, joint targets down) and the HBM bytes the servo call and the
                         chained baseline move, counted from the layouts
  gpu                    name, power limit and SM clock, read in the same run
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

K = 10
LPF_SLOTS = [0, 1, 2, 6, 7, 8, 9, 10, 11]
QH = np.array([0, 0.87, -1.5])


def servo_state(mpc, B):
    """Homing pose as q, its world foot positions (body at the CoM height, Go1 leg geometry via leg FK) as homing, zero filters."""
    import torch
    import quadrupedal_loco_b200 as q
    pos = np.zeros((3, 4)); J = np.zeros((9, 4))
    qh = np.ascontiguousarray(np.tile(QH, (4, 1)).T)
    bp = np.ascontiguousarray(np.tile([0.0, 0.0, 0.309458], (4, 1)).T); br = np.zeros((3, 4))
    mpc.leg_fk_host(4, qh, np.arange(4, dtype=np.int32), bp, br, pos, J)
    s = np.zeros((q.SERVO_STATE_ROWS, B))
    s[q.SERVO_ROW_Q:q.SERVO_ROW_Q + 12] = np.tile(QH, 4)[:, None]
    s[q.SERVO_ROW_HOMING:q.SERVO_ROW_HOMING + 12] = pos.T.reshape(12)[:, None]
    return torch.from_numpy(s).cuda()


def hbm_bytes():
    """Bytes per robot one K-tick call moves in HBM, counted from the layouts (first touch; no cache reuse assumed)."""
    fused = 8 * (11 + 69) + 8 * (12 + 45) + 8 * 12 * K                  # 9 + 2 message slots and the state in, state + q out
    # per tick: lpf reads 9 slots + 45 state, writes 45 state (+ counter only while counting) + 9 out;
    # servo_kin reads com 3 + theta 3 + feet 6 + homing 12 + q 12, writes q 12
    chained = K * 8 * ((9 + 45) + (45 + 9) + (3 + 3 + 6 + 12 + 12) + 12)
    return {"fused": fused, "chained": chained}


def measure(mpc, B, warm, reps, window):
    import torch
    import quadrupedal_loco_b200 as q
    f = gsp.Farm(mpc, 10, B, seed=1000 + B)
    sv = servo_state(mpc, B)
    q_d = torch.zeros(B, 12 * K, dtype=torch.float64, device="cuda")
    q_h = torch.zeros(B, 12 * K, dtype=torch.float64).pin_memory()
    for _ in range(warm):
        f.call()
        mpc.servo_stack_tick(B, K, 102, 1.0, f.state, sv, q_d)
    mpc.synchronize()
    s = torch.cuda.ExternalStream(mpc.stream)
    # the chained baseline on its own copy of the servo state
    coef = np.tile(q.lpf_coefficients(1000.0, 3.0), (9, 1))
    rows9 = torch.tensor(LPF_SLOTS, dtype=torch.int32, device="cuda")
    gait, traj = f.state[q.STACK_ROW_GAIT:q.STACK_ROW_GAIT + 100], f.state[q.STACK_ROW_TRAJ:q.STACK_ROW_TRAJ + 100]
    sv_c = sv.clone()
    cq, hom, lpf = sv_c[0:12].clone(), sv_c[12:24].clone(), sv_c[24:69].clone().view(5, 9, B)
    out9 = torch.zeros(9, B, dtype=torch.float64, device="cuda")
    theta = torch.stack([traj[72], traj[73], torch.zeros_like(traj[72])])
    torch.cuda.synchronize()

    def fused():
        mpc.servo_stack_tick(B, K, 102, 1.0, f.state, sv, q_d)

    def chained():
        for _ in range(K):
            mpc.lpf_batch(B, 9, coef, gait, lpf, out9, in_rows_d=rows9)
            mpc.servo_kin_tick(B, 102, 1.0, out9[0:3], theta, out9[6:9], out9[3:6], hom, cq)

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    t = {"fused": [], "chained": []}
    for _ in range(3):
        fused(); chained()
    mpc.synchronize()
    for _ in range(reps):
        for name, fn in (("fused", fused), ("chained", chained)):
            ev[0].record(s); fn(); ev[1].record(s); ev[1].synchronize()
            t[name].append(ev[0].elapsed_time(ev[1]) * 1e3)
    # gait stack call alone, same schedule position type (fast and planner calls as they come)
    gs = []
    for _ in range(reps):
        ev[0].record(s); f.call(); ev[1].record(s); ev[1].synchronize()
        gs.append(ev[0].elapsed_time(ev[1]) * 1e3)
    # sustained periods: gait stack call + servo call with the joint targets down
    n = 0
    t0 = time.perf_counter()
    while True:
        for _ in range(10):
            f.call()
            mpc.servo_stack_tick(B, K, 102, 1.0, f.state, sv, q_d, q=q_h)
            n += 1
        mpc.synchronize()
        el = time.perf_counter() - t0
        if el >= window:
            break
    med = lambda v: float(np.median(v))
    per_period_s = el / n
    return {
        "B": B, "nh": 10, "K": K, "warm_ticks": warm, "reps": reps,
        "fused_us": {"median": med(t["fused"]), "p10": float(np.percentile(t["fused"], 10)), "p90": float(np.percentile(t["fused"], 90))},
        "chained_us": {"median": med(t["chained"]), "p10": float(np.percentile(t["chained"], 10)),
                       "p90": float(np.percentile(t["chained"], 90))},
        "fused_speedup": med(t["chained"]) / med(t["fused"]),
        "gait_stack_call_us_median": med(gs),
        "period": {"seconds": el, "periods": n, "periods_per_s": n / el, "robot_periods_per_s": B * n / el,
                   "share_of_10ms": per_period_s / 0.010},
        "bytes_per_robot_period": {"h2d": gsp.SENSOR_ROWS * 8, "d2h": 12 * K * 8, "d2h_stack_rows": len(gsp.SLOTS) * 8, "hbm_servo_call": hbm_bytes()["fused"],
                                   "hbm_chained_baseline": hbm_bytes()["chained"]},
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--warm", type=int, default=200, help="fast ticks walked before timing")
    ap.add_argument("--reps", type=int, default=100, help="timed calls per mode")
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
