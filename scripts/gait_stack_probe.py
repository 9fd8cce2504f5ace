"""Gait stack tick (go1mpc_gait_stack_tick_host_async) on a GPU: one JSON line per run.

Setup: B in --batch (default 4096, 65536), nh = 10, every robot walked --warm fast ticks into the gait on the reference's clock
(planner every 25 ms, fast node every 10 ms), then:
  device_us        CUDA events around lone calls, planner calls and fast-only calls separately (median over the schedule)
  host_us          host-to-host p50 / p99 of single calls with pinned buffers (call + stream synchronise)
  sustained        robot-ticks/s and QP solves/s (1 body QP per fast tick, 3 planner QPs more per planner tick) over a window
                   of at least --window s of back-to-back calls, with the call count
  bytes_per_robot_tick  H2D and D2H of the call
  rt_pre_us        rt_pre_kernel from torch.profiler in a separate run at the largest batch (--no-profile skips it)
  gpu              name, power limit and SM clock, read in the same run
The result slots are what a servo consumes: /MPC/Gait 0-2, 6-11, 39-41 and /rtMPC/traj 72-75 (16 doubles per robot).

--dump-outputs DIR runs a fixed seeded schedule (--dump-batch robots, --dump-ticks fast ticks) and writes the sha256 of the whole
state, body records and rows plus a fixed sample of robots (.npy), so two builds can be compared output for output.  With
--via-nodes the same schedule drives go1mpc_nlp_node_tick_batch + go1mpc_rt_node_tick_msgs_batch instead (bit-identical to the
stack), which a library without the stack entry also has: put that build's tree first on PYTHONPATH to dump it."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.append(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))   # after PYTHONPATH: another build's tree may come first

SLOTS = [0, 1, 2, 6, 7, 8, 9, 10, 11, 39, 40, 41, 172, 173, 174, 175]
CTL_SLOTS = [0, 10, 11, 13, 14, 19, 20, 21, 22, 23, 24]
SENSOR_ROWS = 11


def planner_ticks(k):
    return k == 0 or (10 * k) // 25 > (10 * (k - 1)) // 25


def sensors(B, n, seed):
    """n seeded sensor blocks [11][B]: control flag 1, small body angles / rates, foot locations around the nominal stance."""
    rng = np.random.Generator(np.random.Philox(seed))
    out = []
    for _ in range(n):
        s = np.zeros((SENSOR_ROWS, B))
        s[0] = 1.0
        s[1:5] = rng.uniform(-0.03, 0.03, (4, B))
        for base, y in ((5, 0.127), (8, -0.127)):
            s[base] = rng.uniform(-0.02, 0.02, B); s[base + 1] = y + rng.uniform(-0.01, 0.01, B); s[base + 2] = rng.uniform(-0.005, 0.005, B)
        out.append(s)
    return out


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, pl, sm, smax = [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": pl, "sm_clock": sm, "sm_clock_max": smax}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


class Farm:
    """B robots on the stack entry with pinned host buffers."""

    def __init__(self, mpc, nh, B, seed, n_sensors=16):
        import torch
        import quadrupedal_loco_b200 as q
        self.mpc, self.nh, self.B, self.q = mpc, nh, B, q
        col = mpc.gait_stack_default_state(nh)
        self.state = torch.from_numpy(np.repeat(col[:, None], B, axis=1).copy()).cuda()
        self.body_out = torch.zeros(B, q.body_out_stride(nh), dtype=torch.float64, device="cuda")
        self.rows_d = torch.zeros(B, len(SLOTS), dtype=torch.float64, device="cuda")
        self.rows = torch.zeros(B, len(SLOTS), dtype=torch.float64).pin_memory()
        self.sens = [torch.from_numpy(s).pin_memory() for s in sensors(B, n_sensors, seed)]
        self.t = [[mpc.gait_stack_tick_struct(nh, pl, s, self.state, self.body_out, SLOTS, self.rows_d, self.rows) for s in self.sens]
                  for pl in (0, 1)]
        self.k = 0
        torch.cuda.synchronize()

    def call(self, k=None):
        k = self.k if k is None else k
        pl = planner_ticks(k)
        self.mpc.gait_stack_tick_host_async(self.B, self.t[pl][k % len(self.sens)], None)
        self.k = k + 1
        return pl


def measure(mpc, nh, B, warm, window, reps):
    import torch
    f = Farm(mpc, nh, B, seed=1000 + B)
    for _ in range(warm):
        f.call()
    mpc.synchronize()
    s = torch.cuda.ExternalStream(mpc.stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dev = {0: [], 1: []}
    host = {0: [], 1: []}
    for _ in range(reps):
        e0.record(s); pl = f.call(); e1.record(s); e1.synchronize()
        dev[pl].append(e0.elapsed_time(e1) * 1e3)
    for _ in range(reps):
        t0 = time.perf_counter(); pl = f.call(); mpc.synchronize(); host[pl].append((time.perf_counter() - t0) * 1e6)
    n, npl = 0, 0
    t0 = time.perf_counter()
    while True:
        for _ in range(10):
            npl += f.call(); n += 1
        mpc.synchronize()
        el = time.perf_counter() - t0
        if el >= window:
            break
    pct = lambda v, p: float(np.percentile(v, p)) if v else None
    return {
        "B": B, "nh": nh, "warm_ticks": warm,
        "device_us": {"planner_call_median": pct(dev[1], 50), "fast_call_median": pct(dev[0], 50),
                      "planner_calls": len(dev[1]), "fast_calls": len(dev[0])},
        "host_us": {"planner_p50": pct(host[1], 50), "planner_p99": pct(host[1], 99), "fast_p50": pct(host[0], 50),
                    "fast_p99": pct(host[0], 99), "planner_calls": len(host[1]), "fast_calls": len(host[0])},
        "sustained": {"seconds": el, "calls": n, "planner_calls": npl, "robot_ticks_per_s": B * n / el,
                      "qp_solves_per_s": B * (n + 3 * npl) / el},
        "bytes_per_robot_tick": {"h2d": SENSOR_ROWS * 8, "d2h": len(SLOTS) * 8},
    }


def profile_rt_pre(mpc, nh, B, warm, calls, outdir):
    import torch
    from torch.profiler import ProfilerActivity, profile
    f = Farm(mpc, nh, B, seed=2000 + B)
    for _ in range(warm):
        f.call()
    mpc.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            f.call()
        mpc.synchronize()
    per = {}
    for ka in prof.key_averages():
        tot = getattr(ka, "self_device_time_total", None)
        if tot is None:
            tot = getattr(ka, "self_cuda_time_total", 0.0)
        if tot and ka.count:
            per[ka.key.split("(")[0].split("::")[-1]] = {"count": int(ka.count), "mean_us": float(tot) / ka.count}
    if outdir:
        prof.export_chrome_trace(os.path.join(outdir, f"gait_stack_b{B}.pt.trace.json"))
    return {"B": B, "calls": calls, "rt_pre_us": per.get("rt_pre_kernel", {}).get("mean_us"), "kernels": per}


def dump(mpc, nh, B, ticks, outdir, via_nodes):
    """Fixed seeded schedule from the default state; writes digests + a robot sample."""
    import torch
    import quadrupedal_loco_b200 as q
    sens = sensors(B, 8, 4242)
    nlp_n = mpc.nlp_node_state_doubles()
    if via_nodes:
        nlp = torch.from_numpy(np.repeat(mpc.nlp_node_default_state()[:, None], B, axis=1).copy()).cuda()
        rt = torch.from_numpy(np.repeat(mpc.rt_node_default_state(nh)[:, None], B, axis=1).copy()).cuda()
        gait = torch.zeros(100, B, dtype=torch.float64, device="cuda"); traj = torch.zeros_like(gait)
        r2n = torch.zeros(25, B, dtype=torch.float64, device="cuda"); ctl = torch.zeros_like(r2n)
        body_in = torch.zeros(B, q.body_in_stride(nh), dtype=torch.float64, device="cuda")
        body_out = torch.zeros(B, q.body_out_stride(nh), dtype=torch.float64, device="cuda")
        wd = torch.zeros(B, dtype=torch.int32, device="cuda")
        sens_d = [torch.from_numpy(s).cuda() for s in sens]
        torch.cuda.synchronize()
        with torch.cuda.stream(torch.cuda.ExternalStream(mpc.stream)):
            for k in range(ticks):
                if planner_ticks(k):
                    wd += 1
                    mpc.nlp_node_tick(B, nlp, wd, gait, rfoot_fb_d=r2n[22:25], lfoot_fb_d=r2n[19:22])
                ctl[CTL_SLOTS] = sens_d[k % len(sens)]
                mpc.rt_node_tick_msgs(nh, B, rt, gait, ctl, body_in, body_out, traj, r2n)
            state = torch.cat([nlp, gait, r2n, wd[None].double(), traj, rt])
            rows = torch.cat([gait, traj])[SLOTS].T.contiguous()
        mpc.synchronize(); torch.cuda.synchronize()
    else:
        f = Farm(mpc, nh, B, seed=0, n_sensors=1)
        f.sens = [torch.from_numpy(s).pin_memory() for s in sens]
        f.t = [[mpc.gait_stack_tick_struct(nh, pl, s, f.state, f.body_out, SLOTS, f.rows_d, f.rows) for s in f.sens] for pl in (0, 1)]
        for k in range(ticks):
            f.call(k)
        mpc.synchronize(); torch.cuda.synchronize()
        state, body_out, rows = f.state, f.body_out, f.rows_d
    assert state.shape[0] == nlp_n + 226 + mpc.rt_node_state_doubles(nh)
    os.makedirs(outdir, exist_ok=True)
    sample = np.sort(np.random.Generator(np.random.Philox(7)).choice(B, min(B, 256), replace=False))
    out = {}
    for name, t in (("state", state), ("body_out", body_out), ("rows", rows)):
        a = t.cpu().numpy()
        out[name] = hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
        np.save(os.path.join(outdir, name + ".npy"), a[:, sample] if name == "state" else a[sample])
    np.save(os.path.join(outdir, "robot.npy"), sample)
    out.update(B=B, nh=nh, ticks=ticks, via_nodes=bool(via_nodes), library=q.library_path())
    with open(os.path.join(outdir, "digest.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--nh", type=int, default=10)
    ap.add_argument("--warm", type=int, default=200, help="fast ticks walked before timing")
    ap.add_argument("--reps", type=int, default=100, help="lone calls per timing mode")
    ap.add_argument("--window", type=float, default=0.5, help="seconds of back-to-back calls (>= 0.2)")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--trace-dir", default=None, help="write the torch.profiler trace here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR")
    ap.add_argument("--dump-batch", type=int, default=65536)
    ap.add_argument("--dump-ticks", type=int, default=300)
    ap.add_argument("--via-nodes", action="store_true")
    a = ap.parse_args()
    import quadrupedal_loco_b200 as q
    mpc = q.Go1Mpc(0)
    res = {"gpu": gpu_info(), "slots": SLOTS}
    if a.dump_outputs:
        res["dump"] = dump(mpc, a.nh, a.dump_batch, a.dump_ticks, a.dump_outputs, a.via_nodes)
    else:
        assert a.window >= 0.2
        res["runs"] = [measure(mpc, a.nh, B, a.warm, a.window, a.reps) for B in a.batch]
        if not a.no_profile:
            res["profile"] = profile_rt_pre(mpc, a.nh, max(a.batch), a.warm, 20, a.trace_dir)
        res["gpu_after"] = gpu_info()
    mpc.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
