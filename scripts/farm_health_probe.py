"""Cost of the farm health counters on a GPU: wall time per device-fed 10 ms period with and without health, one JSON line.

Setup per batch B (--batch, default 4096 65536): scripts/farm_device_inputs_probe.py's farm (nh = 10, gait mode 102, K = 10,
clocks spread over c mod 5, a plant of two device copies per period writing the sensor rows and the restart index).  A period is
restore (go1mpc_farm_copy_async from a bank of 16 freshly reset robots; the index restarts about 1 % of the robots per period)
-> clocked tick -> torque tick, every input on the device, captured once per mode and replayed back to back with the plant
between replays and one synchronisation at the end of each window:
  plain    go1mpc_gait_stack_tick_clocked_async + go1mpc_servo_torque_tick_async, farm copy without health blocks
  health   go1mpc_gait_stack_tick_clocked_health_async + go1mpc_servo_torque_tick_health_async, health_d on both sides of the copy
The two modes run on two farms walked through the same warm-up, alternated over --rounds windows of --periods periods; reported
per mode: the per-period time of each window, their median, and health / plain - 1.  profile: one torch.profiler run per mode
(B = the first batch) with the GPU time of each kernel of one replayed period.  gpu: name, power limit and SM clock, read in the
same run before and after.
"""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.append(os.path.dirname(HERE))
sys.path.append(HERE)
import farm_device_inputs_probe as fdp  # noqa: E402
import gait_stack_probe as gsp  # noqa: E402

NH, K, GM, YC = fdp.NH, fdp.K, fdp.GM, fdp.YC
BANK = 16


class Farm(fdp.Farm):
    """fdp.Farm plus a bank of freshly reset robots, a restart index written by the plant and (with health) the counters."""

    def __init__(self, mpc, B, seed, with_health):
        import torch
        import quadrupedal_loco_b200 as q
        super().__init__(mpc, B, seed)
        dev = torch.device("cuda", 0)
        self.health = torch.zeros(q.HEALTH_ROWS, B, dtype=torch.int32, device=dev) if with_health else None
        col = mpc.gait_stack_default_state(NH)
        self.bank = dict(state=torch.from_numpy(np.repeat(col[:, None], BANK, axis=1).copy()).to(dev),
                         body_out=torch.zeros(BANK, q.body_out_stride(NH), dtype=torch.float64, device=dev),
                         clock=torch.zeros(BANK, dtype=torch.int32, device=dev),
                         servo=self.servo[:, :BANK].clone(), force=torch.zeros(q.SERVO_FORCE_ROWS, BANK, dtype=torch.float64, device=dev),
                         health=torch.zeros(q.HEALTH_ROWS, BANK, dtype=torch.int32, device=dev) if with_health else None)
        b = np.arange(B)
        self.index_table = torch.from_numpy(np.stack([np.where((b + j) % 100 == 0, (b + j) % BANK, -1) for j in range(100)])
                                            .astype(np.int32)).to(dev)
        self.index_d = torch.full((B,), -1, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()

    def plant(self):
        import torch
        with torch.cuda.stream(self.s):
            self.sensor_d.copy_(self.sens_table[self.j % 16])
            self.index_d.copy_(self.index_table[self.j % 100])
            self.reset_d.zero_()                              # the warm-up's reset periods set their own flags after this
        self.j += 1

    def restore_period(self):
        m, k = self.mpc, self.bank
        dst = m.farm_columns(self.B, self.state, self.body_out, self.clock, self.servo, self.force, self.health)
        src = m.farm_columns(BANK, k["state"], k["body_out"], k["clock"], k["servo"], k["force"], k["health"])
        m.farm_copy(NH, dst, src, self.index_d, stream=self.st)
        t = m.gait_stack_tick_clocked_struct(NH, None, self.clock, self.state, self.body_out, gsp.SLOTS, self.rows_d, sensor_d=self.sensor_d)
        m.gait_stack_tick_clocked_async(self.B, t, self.st, health_d=self.health)
        m.servo_torque_tick(self.B, K, GM, 1.0, YC, self.state, self.servo, self.force, self.meas, self.q_d, self.tau_d, stream=self.st,
                            health_d=self.health)

    def capture_restore(self):
        import ctypes
        m = self.mpc
        m._check(m.lib.go1mpc_graph_capture_begin(m.h, self.st), "capture_begin")
        self.restore_period()
        ge = ctypes.c_void_p()
        m._check(m.lib.go1mpc_graph_capture_end(m.h, self.st, ctypes.byref(ge)), "capture_end")
        return ge


def walk(f, periods):
    fdp.warm_up(f, periods)                                   # spread clocks, walk into the gait
    for _ in range(3):                                        # both forms of the restore period warmed up on the stream
        f.plant()
        f.restore_period()
    f.s.synchronize()


def measure(mpc, B, P, rounds, warm):
    import torch
    farms = {m: Farm(mpc, B, 2000 + B, m == "health") for m in ("plain", "health")}
    for f in farms.values():
        walk(f, warm)
    graphs = {m: f.capture_restore() for m, f in farms.items()}
    per = {m: [] for m in farms}
    try:
        for m, f in farms.items():
            fdp.timed(f, 5, lambda: (f.plant(), f.launch(graphs[m])))
        for _ in range(rounds):
            for m, f in farms.items():
                per[m].append(fdp.timed(f, P, lambda: (f.plant(), f.launch(graphs[m]))))
    finally:
        for m, f in farms.items():
            f.s.synchronize()
            f.destroy(graphs[m])
    res = {"B": B, "nh": NH, "K": K, "gait_mode": GM, "periods": P, "rounds": rounds, "warm_periods": warm,
           "clock_residues": np.bincount(farms["plain"].clock.cpu().numpy() % 5, minlength=5).tolist(),
           "restarts_per_period_mean": (farms["plain"].index_table >= 0).sum(dim=1).float().mean().item()}
    for m in farms:
        res[m] = {"us_per_period_median": float(np.median(per[m])), "us_per_period_rounds": per[m]}
    res["health_over_plain_minus_1"] = res["health"]["us_per_period_median"] / res["plain"]["us_per_period_median"] - 1
    h = farms["health"].health.cpu().numpy()
    res["health_rows_sum"] = h[:-1].sum(axis=1).tolist()
    del farms
    torch.cuda.empty_cache()
    return res


def profile(mpc, B, out_dir):
    """GPU time per kernel of one replayed period in each mode (torch.profiler)."""
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile
    res = {"B": B}
    for m in ("plain", "health"):
        f = Farm(mpc, B, 3000 + B, m == "health")
        walk(f, 10)
        ge = f.capture_restore()
        try:
            f.s.synchronize()
            with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                f.plant(); f.launch(ge)
                f.s.synchronize()
            ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
            kern = {}
            for e in ev:
                kern[e.name] = kern.get(e.name, 0.0) + getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0))
            res[m] = {"kernels_us": {k: round(v, 2) for k, v in sorted(kern.items(), key=lambda kv: -kv[1])}, "gpu_events": len(ev)}
            if out_dir:
                prof.export_chrome_trace(os.path.join(out_dir, f"farm_health_{m}.pt.trace.json"))
        finally:
            f.s.synchronize()
            f.destroy(ge)
        del f
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--periods", type=int, default=200, help="periods per timed window")
    ap.add_argument("--rounds", type=int, default=5, help="timed windows per mode, modes alternated")
    ap.add_argument("--warm", type=int, default=40, help="periods walked before timing")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file (profiler traces beside it)")
    a = ap.parse_args()
    import quadrupedal_loco_b200 as q
    out_dir = os.path.dirname(os.path.abspath(a.out)) if a.out else None
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
    mpc = q.Go1Mpc(0)
    res = {"gpu": gsp.gpu_info(), "runs": [measure(mpc, B, a.periods, a.rounds, a.warm) for B in a.batch]}
    res["profile"] = profile(mpc, a.batch[0], out_dir)
    res["gpu_after"] = gsp.gpu_info()
    mpc.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
