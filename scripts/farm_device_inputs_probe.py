"""Device-fed farm periods on a GPU: wall time per 10 ms period of a farm closed through a simulator, one JSON line per run.

Setup per batch B (--batch, default 1024 4096 65536): nh = 10, gait mode 102, K = 10 servo ticks, clocks spread over c mod 5
(robots with b mod 5 = i reset in warm-up period i), about 1 % of the robots reset every period (b + period = 0 mod 100), and a
trivial plant: two device copies per period that write the next sensor rows (16 seeded blocks in rotation) and the next reset
flags, standing in for a simulator's kernel.  A period is reset -> clocked tick -> torque tick; rows, q and tau stay on the
device.  Modes, each timed over --periods consecutive periods with a host clock that stops after a final synchronisation:
  a_host_fed_graph      today's form: the period captured with pinned sensor / reset buffers; every period the plant runs, its
                        outputs come down into the pinned buffers, the stream is synchronised and the graph replayed
  b_device_fed_graph    the period captured with sensor_d / reset_d, replayed back to back with the plant enqueued between
                        replays, one synchronisation at the end
  c_device_fed_direct   the device-fed period enqueued call by call, back to back, one synchronisation at the end
The modes are alternated over --rounds rounds; reported per mode: the per-period time of each round and their median.
profile: a separate torch.profiler run (B = the second batch) of one device-fed period (direct calls, then one replay) and of one
host-fed period, with the count of host-to-device and device-to-host copies in each.  gpu: name, power limit and SM clock, read
in the same run before and after.
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.append(os.path.dirname(HERE))
sys.path.append(HERE)
import gait_stack_probe as gsp  # noqa: E402
import servo_stack_probe as ssp  # noqa: E402

NH, K, GM, YC = 10, 10, 102, 0.9
Q0 = np.tile(ssp.QH, 4)


class Farm:
    """B robots: gait stack, clocks, servo and force state, plant outputs on the device and pinned host copies of them."""

    def __init__(self, mpc, B, seed):
        import torch
        import quadrupedal_loco_b200 as q
        dev = torch.device("cuda", 0)
        self.mpc, self.B = mpc, B
        self.s = torch.cuda.Stream()
        self.st = self.s.cuda_stream
        col = mpc.gait_stack_default_state(NH)
        self.state = torch.from_numpy(np.repeat(col[:, None], B, axis=1).copy()).to(dev)
        self.body_out = torch.zeros(B, q.body_out_stride(NH), dtype=torch.float64, device=dev)
        self.rows_d = torch.zeros(B, len(gsp.SLOTS), dtype=torch.float64, device=dev)
        self.clock = torch.zeros(B, dtype=torch.int32, device=dev)
        self.servo = ssp.servo_state(mpc, B)
        self.force = torch.zeros(q.SERVO_FORCE_ROWS, B, dtype=torch.float64, device=dev)
        self.meas = torch.from_numpy(np.ascontiguousarray(np.repeat(np.concatenate([Q0, np.zeros(12)])[:, None], B, axis=1))).to(dev)
        self.q_d = torch.zeros(B, 12 * K, dtype=torch.float64, device=dev)
        self.tau_d = torch.zeros(B, 12 * K, dtype=torch.float64, device=dev)
        # the plant's tables and outputs
        self.sens_table = torch.from_numpy(np.stack(gsp.sensors(B, 16, seed))).to(dev)
        b = np.arange(B)
        self.flag_table = torch.from_numpy(np.stack([((b + j) % 100 == 0) for j in range(100)]).astype(np.int32)).to(dev)
        self.stagger = torch.from_numpy(np.stack([(b % 5 == i) for i in range(5)]).astype(np.int32)).to(dev)
        self.sensor_d = torch.zeros(gsp.SENSOR_ROWS, B, dtype=torch.float64, device=dev)
        self.reset_d = torch.zeros(B, dtype=torch.int32, device=dev)
        self.sensor_h = torch.zeros(gsp.SENSOR_ROWS, B, dtype=torch.float64).pin_memory()
        self.reset_h = torch.zeros(B, dtype=torch.int32).pin_memory()
        self.j = 0
        torch.cuda.synchronize()

    def plant(self):
        """The simulator's step: the next sensor rows and reset flags, on the farm's stream."""
        import torch
        with torch.cuda.stream(self.s):
            self.sensor_d.copy_(self.sens_table[self.j % 16])
            self.reset_d.copy_(self.flag_table[self.j % 100])
        self.j += 1

    def period(self, device):
        m = self.mpc
        kw = dict(reset_d=self.reset_d) if device else dict(reset=self.reset_h)
        r = m.gait_stack_reset_struct(NH, kw.get("reset"), self.clock, self.state, self.body_out, self.servo, Q0,
                                      reset_d=kw.get("reset_d"))
        m.gait_stack_reset_async(self.B, r, self.st)
        sensor, sensor_d = (None, self.sensor_d) if device else (self.sensor_h, None)
        t = m.gait_stack_tick_clocked_struct(NH, sensor, self.clock, self.state, self.body_out, gsp.SLOTS, self.rows_d,
                                             sensor_d=sensor_d)
        m.gait_stack_tick_clocked_async(self.B, t, self.st)
        m.servo_torque_tick(self.B, K, GM, 1.0, YC, self.state, self.servo, self.force, self.meas, self.q_d, self.tau_d, stream=self.st,
                            **kw)

    def download(self):
        """Host-fed form: the plant's outputs into the pinned buffers, then wait for the stream."""
        with_stream(self.s, lambda: (self.sensor_h.copy_(self.sensor_d, non_blocking=True),
                                     self.reset_h.copy_(self.reset_d, non_blocking=True)))
        self.s.synchronize()

    def capture(self, device):
        m = self.mpc
        m._check(m.lib.go1mpc_graph_capture_begin(m.h, self.st), "capture_begin")
        self.period(device)
        ge = ctypes.c_void_p()
        m._check(m.lib.go1mpc_graph_capture_end(m.h, self.st, ctypes.byref(ge)), "capture_end")
        return ge

    def launch(self, ge):
        self.mpc._check(self.mpc.lib.go1mpc_graph_launch(self.mpc.h, ge, self.st), "graph_launch")

    def destroy(self, ge):
        self.mpc._check(self.mpc.lib.go1mpc_graph_destroy(self.mpc.h, ge), "graph_destroy")


def with_stream(s, fn):
    import torch
    with torch.cuda.stream(s):
        return fn()


def warm_up(f, periods):
    """Spread the clocks over c mod 5 and walk the farm into the gait, both forms of every call included."""
    for p in range(periods):
        f.plant()
        if p < 5:
            with_stream(f.s, lambda: f.reset_d.copy_(f.stagger[p]))
        f.download()
        f.period(device=p % 2 == 0)
    f.s.synchronize()


def timed(f, P, step):
    f.s.synchronize()
    t0 = time.perf_counter()
    for _ in range(P):
        step()
    f.s.synchronize()
    return (time.perf_counter() - t0) * 1e6 / P


def measure(mpc, B, P, rounds, warm):
    import torch
    f = Farm(mpc, B, seed=2000 + B)
    warm_up(f, warm)
    residues = np.bincount(f.clock.cpu().numpy() % 5, minlength=5).tolist()
    g_host, g_dev = f.capture(False), f.capture(True)
    res = {"B": B, "nh": NH, "K": K, "gait_mode": GM, "periods": P, "rounds": rounds, "warm_periods": warm, "clock_residues": residues}
    modes = {
        "a_host_fed_graph": lambda: (f.plant(), f.download(), f.launch(g_host)),
        "b_device_fed_graph": lambda: (f.plant(), f.launch(g_dev)),
        "c_device_fed_direct": lambda: (f.plant(), f.period(True)),
    }
    per = {m: [] for m in modes}
    try:
        for m, step in modes.items():                                      # one untimed pass of each mode
            timed(f, 5, step)
        for _ in range(rounds):
            for m, step in modes.items():
                per[m].append(timed(f, P, step))
    finally:
        f.s.synchronize()
        f.destroy(g_host); f.destroy(g_dev)
    flags = f.flag_table.sum(dim=1).float().mean().item()
    for m in modes:
        res[m] = {"us_per_period_median": float(np.median(per[m])), "us_per_period_rounds": per[m]}
    res["resets_per_period_mean"] = flags
    res["a_over_b"] = res["a_host_fed_graph"]["us_per_period_median"] / res["b_device_fed_graph"]["us_per_period_median"]
    del f
    torch.cuda.empty_cache()
    return res


def profile(mpc, B, out_dir):
    """Copies listed by torch.profiler in one device-fed period (direct, then one graph replay) and in one host-fed period."""
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile
    f = Farm(mpc, B, seed=3000 + B)
    warm_up(f, 10)
    g_dev, g_host = f.capture(True), f.capture(False)
    res = {"B": B}
    try:
        for name, step in (("device_fed_period", lambda: (f.plant(), f.period(True), f.plant(), f.launch(g_dev))),
                           ("host_fed_period", lambda: (f.plant(), f.download(), f.launch(g_host)))):
            f.s.synchronize()
            with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                step()
                f.s.synchronize()
            ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
            names = sorted({e.name for e in ev})
            res[name] = {"htod": sum("HtoD" in e.name for e in ev), "dtoh": sum("DtoH" in e.name for e in ev),
                         "dtod": sum("DtoD" in e.name for e in ev), "gpu_events": len(ev), "event_names": names}
            if out_dir:
                prof.export_chrome_trace(os.path.join(out_dir, f"farm_device_inputs_{name}.pt.trace.json"))
    finally:
        f.s.synchronize()
        f.destroy(g_dev); f.destroy(g_host)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, nargs="+", default=[1024, 4096, 65536])
    ap.add_argument("--periods", type=int, default=200, help="periods per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="timed windows per mode, modes alternated")
    ap.add_argument("--warm", type=int, default=40, help="periods walked before timing")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file (profiler traces beside it)")
    a = ap.parse_args()
    import quadrupedal_loco_b200 as q
    out_dir = os.path.dirname(os.path.abspath(a.out)) if a.out else None
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
    mpc = q.Go1Mpc(0)
    res = {"gpu": gsp.gpu_info(), "runs": [measure(mpc, B, a.periods, a.rounds, a.warm) for B in a.batch]}
    res["profile"] = profile(mpc, a.batch[min(1, len(a.batch) - 1)], out_dir)
    res["gpu_after"] = gsp.gpu_info()
    mpc.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
