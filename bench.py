#!/usr/bin/env python
"""bench.py -- throughput of the batched Go1 MPC QP hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W                    (own arm; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W   (CPU arm, host cores)

A "step" is one pass of the Go1 MPC hot path over one batch of synthetic robots: per robot one
step-location/step-timing SQP tick (3 QP solves, n=4 p=1 m=24, plus write-back, LIPM roll-out and step
indices) followed by one body-inclination MPC tick (condensation -> Goldfarb-Idnani QP -> clamp ->
roll-out; 1 QP solve, n=2nh m=12nh).  `value` counts QP solves (one solve = one solve_quadprog call of
the reference).

Workloads (SURVEY.md section 8d):
  cfg3 (default; the configuration BASELINE.json quotes at 1/2/4/8 GPUs): GLOBAL batch 65536 robots,
       sharded contiguously over the N ranks (strong scaling, no collective inside the step), planner
       and body MPC with the feedback-gain presets the reference ships commented out
       (NLPClass_sqp.cpp:986-993, PRMPCClass.cpp:681-687), state perturbations 2x cfg2, seed 0xB2000003.
  cfg2 (--config cfg2): 4096 robots PER GPU (weak scaling), gains 0 as shipped, seed 0xB2000002 + rank.

Timing: CUDA events on the launching stream, W untimed warm-up steps, then exactly K timed steps
bracketed by barrier + synchronize; max over ranks.  The K steps are independent robot batches dealt
round-robin over a few streams; the whole K-step schedule is captured ONCE into a CUDA graph before the
timed region (go1mpc_graph_capture_*), so the timed region is one graph launch: no host enqueue, no
thread start-up inside it, and `--steps 20` measures the same thing as `--steps 2000`.  Steps rotate
through enough distinct input batches that the footprint exceeds 2x L2 (126 MB).
The `e2e` leg calls go1mpc_control_tick_host_async with pinned HOST buffers (H2D of the tick's
arguments, both ticks, compact result rows) and, for N > 1, gathers the result rows of every rank to
rank 0 over NCCL once per batch; rank 0 reads the gathered rows back to host memory.

--dump-outputs DIR writes what the last timed step computed (see dump_outputs) so that two builds can be compared
output for output: the inputs depend only on the arguments.  The run writes nothing else to disk outside a
temporary directory, so it can run from a read-only tree.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True           # no __pycache__ in the tree the bench runs from

METRIC = "batched MPC QP solves/sec"
UNIT = "solves/s"
L2_BYTES = 126 * 1024 * 1024
PRESET_STEP_LAMDA = (0.25, 0.001, 0.025, 0.001)     # NLPClass_sqp.cpp:986-993 (commented preset)
# planner workload mix (synth.step_timing_inputs): forward-walking periods, pushes sized so that the benched QPs are mostly
# feasible (> 99 % at cfg2's amplitude, ~93 % at cfg3's 2x)
PLANNER_MIX = dict(push_x=0.4, push_y=0.75, p_hi=16)
PRESET_BODY_LAMDA = (0.2, 0.001, 0.2, 0.001)        # PRMPCClass.cpp:681-687 (commented preset)
SENSOR_ROWS = 10       # e2e: planner input rows uploaded per tick (Go1ControlTick.step_in_rows)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg3", choices=["cfg3", "cfg2"])
    ap.add_argument("--batch", type=int, default=0, help="cfg3: GLOBAL batch (default 65536); cfg2: robots per GPU (default 4096)")
    ap.add_argument("--nh", type=int, default=10, help="body-MPC horizon")
    ap.add_argument("--lanes", type=int, default=0, help="streams the steps are dealt over (0 = by batch size)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="enqueue the timed steps from the host instead of one graph launch")
    ap.add_argument("--latency-samples", type=int, default=1000)
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="e2e, N > 1: how the result rows reach rank 0 -- NVLink peer-memory stores + flags (csrc/peer_gather.cu) or torch.distributed.gather")
    ap.add_argument("--e2e-no-graph", action="store_true", help="e2e: enqueue every step's calls from the host instead of replaying one captured graph per batch slot")
    ap.add_argument("--e2e-no-gather", action="store_true", help="DIAGNOSTIC: leave the gather to rank 0 out of the e2e leg (the number is then not the e2e metric)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (float64; a fixed sample of the robots when "
                         "they exceed 64 MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 arm")
    return a


DUMP_BYTES = 63 * 10 ** 6      # --dump-outputs: data of all files of all ranks, under 64 MB with the .npy headers
DUMP_SEED = 0xB2000D


def dump_outputs(path, rows, first, budget, suffix=""):
    """Writes the per-robot results of one step, rows = {name: [B, k] host array}, as path/<name><suffix>.npy in float64
    (the int diagnostics convert exactly), plus robot<suffix>.npy: the robots' indices in the global batch (first = index
    of row 0).  All B robots when they fit in `budget` bytes, else a sorted sample drawn with the fixed DUMP_SEED."""
    B = len(next(iter(rows.values())))
    per_robot = 8 * (1 + sum(v.shape[1] for v in rows.values()))
    n = min(B, budget // per_robot)
    idx = np.arange(B) if n == B else np.sort(np.random.default_rng(DUMP_SEED).choice(B, n, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, f"robot{suffix}.npy"), (first + idx).astype(np.float64))
    for name, v in rows.items():
        np.save(os.path.join(path, f"{name}{suffix}.npy"), np.ascontiguousarray(v[idx], dtype=np.float64))


def shard_range(B, rank, world):
    per = -(-B // world)
    lo = min(B, rank * per)
    return lo, min(B, lo + per)


def plan(a, world):
    """Batch geometry of the chosen config."""
    if a.config == "cfg3":
        Bg = a.batch or 65536
        return dict(name="cfg3", B_global=Bg, scaling="strong", amp=2.0, scale=2.0, step_lamda=PRESET_STEP_LAMDA,
                    body_lamda=PRESET_BODY_LAMDA, seed="0xB2000003")
    Bl = a.batch or 4096
    return dict(name="cfg2", B_global=Bl * world, scaling="weak", amp=1.0, scale=1.0, step_lamda=(0, 0, 0, 0),
                body_lamda=(0, 0, 0, 0), seed="0xB2000002+rank")


def workload_config(a, world):
    p = plan(a, world)
    per = -(-p["B_global"] // world)
    return {"workload": (f"{p['name']}: Go1 MPC, global batch {p['B_global']} robots ({per} per GPU, batch sharded contiguously over "
                         f"{world} GPU(s), {p['scaling']} scaling); per robot and step: one step-location/step-timing SQP tick (3 QP solves, "
                         f"n=4 p=1 m=24) then one body-inclination MPC tick at horizon {a.nh} (1 QP solve, n={2 * a.nh} m={12 * a.nh}); "
                         + ("feedback-gain presets of the reference (planner 0.25/0.001/0.025/0.001, body 0.2/0.001/0.2/0.001), "
                            "state perturbations 2x cfg2 (body angle kept inside the +-10 deg constraint envelope)" if p["name"] == "cfg3" else "gains 0 as shipped")),
            "batch_per_gpu": per, "global_batch": p["B_global"], "horizon": a.nh, "sqp_iterations": 3,
            "qp_shapes": [[2 * a.nh, 0, 12 * a.nh], [4, 1, 24]], "seed": p["seed"],
            "parallelism": f"batch-sharded x{world}, no collective inside the step; e2e: one gather of the result rows to rank 0 per batch",
            "l2": "inputs rotate through distinct batches totalling > 2x L2 (no flush needed)"}


def make_inputs(a, rank, world, nrot, step_default_state):
    """Per-rank synthetic inputs for `nrot` distinct batches.  cfg3: slot s is the rank's contiguous slice of the global
    batch generated with seed 0xB2000003 + 1000 s, so the robots (and their results) do not depend on N."""
    from quadrupedal_loco_b200 import synth
    p = plan(a, world)
    nh = a.nh
    body, tick, st, sin = [], [], [], []
    for s in range(nrot):
        if p["name"] == "cfg3":
            lo, hi = shard_range(p["B_global"], rank, world)
            d = synth.body_mpc_inputs(p["B_global"], nh, seed=synth.SEED_CFG3 + 1000 * s, scale=p["scale"], theta_clip=0.16)
            d = {k: v[lo:hi] for k, v in d.items()}
            t, x, i = synth.step_timing_inputs(p["B_global"], step_default_state, seed=synth.SEED_CFG3 + 1000 * s, amp=p["amp"], **PLANNER_MIX)
            t, x, i = t[lo:hi], x[lo:hi], i[lo:hi]
        else:
            Bl = p["B_global"] // world
            d = synth.body_mpc_inputs(Bl, nh, seed=synth.SEED_CFG2 + rank + 1000 * s)
            t, x, i = synth.step_timing_inputs(Bl, step_default_state, seed=synth.SEED_CFG2 + rank + 1000 * s, **PLANNER_MIX)
        # planner feedback inputs: the "estimated" CoM state the gains blend in = the planner's own state plus noise
        if any(p["step_lamda"]):
            rng = np.random.Generator(np.random.Philox(77 + s))
            i = i.copy()
            i[:, 0] = x[:, 189] + rng.uniform(-0.01, 0.01, len(t)); i[:, 1] = x[:, 190] + rng.uniform(-0.05, 0.05, len(t))
            i[:, 3] = x[:, 192] + rng.uniform(-0.01, 0.01, len(t)); i[:, 4] = x[:, 193] + rng.uniform(-0.05, 0.05, len(t))
        body.append(d); tick.append(t); st.append(x); sin.append(i)
    return body, tick, st, sin


# ----------------------------------------------------------------------------- CPU arm
def cpu_pool(a, threads, nrobots=None):
    """Native thread pool (oracle/mt_pool.c) over the first `nrobots` robots of rank 0's slot-0 batch at N = 1.
    Returns (run(passes) -> seconds, solves per pass, close)."""
    from tests import oracle_lib
    orc = oracle_lib.Oracle(fast=True)
    lib = orc.lib
    p = plan(a, 1)
    nh = a.nh
    scfg = orc.step_cfg(3, lamda=p["step_lamda"])
    bcfg = orc.body_cfg(nh)
    for k in range(4):
        bcfg.lamda[k] = p["body_lamda"][k]
    body, tick, st, sin = make_inputs(a, 0, 1, 1, orc.step_default_state(scfg))
    d, tick, st, sin = body[0], tick[0], st[0], sin[0]
    B = len(tick) if nrobots is None else min(nrobots, len(tick))
    keep = dict(btick=np.ascontiguousarray(d["tick"][:B], np.int32), tx=np.ascontiguousarray(d["tx"][:B]),
                theta=np.ascontiguousarray(d["theta"][:B]), bstate=np.ascontiguousarray(d["bstate"][:B]),
                refs=np.ascontiguousarray(d["refs"][:B].reshape(B, 9 * nh)), stick=np.ascontiguousarray(tick[:B], np.int32),
                st=np.ascontiguousarray(st[:B]), sin=np.ascontiguousarray(sin[:B]))
    vp = ctypes.c_void_p
    lib.orc_pool_create.restype = vp
    lib.orc_pool_create.argtypes = [ctypes.c_int, vp, vp, ctypes.c_int] + [vp] * 8
    lib.orc_pool_run.restype = ctypes.c_double
    lib.orc_pool_run.argtypes = [vp, ctypes.c_int]
    lib.orc_pool_destroy.argtypes = [vp]
    P = lambda x: x.ctypes.data
    pool = lib.orc_pool_create(threads, ctypes.addressof(bcfg), ctypes.addressof(scfg), B, P(keep["btick"]), P(keep["tx"]), P(keep["theta"]),
                               P(keep["bstate"]), P(keep["refs"]), P(keep["stick"]), P(keep["st"]), P(keep["sin"]))
    assert pool, "orc_pool_create failed"
    _, dg = orc.step_tick_batch(scfg, tick[:512], st[:512].copy(), sin[:512])
    solves = B + int(round(dg[:, 4].mean() * B))

    def run(passes):
        return float(lib.orc_pool_run(pool, passes))

    def close():
        lib.orc_pool_destroy(pool)
        keep.clear()
    return run, solves, close, B


def cpu_baseline(a, budget_s=8.0):
    cores = os.cpu_count() or 1
    out = {}
    for label, thr, nrob in (("1thread", 1, 8192), ("all", cores, None)):
        run, solves, close, B = cpu_pool(a, thr, nrob)
        t1 = run(1)
        n = int(max(1, min(400, budget_s / max(t1, 1e-6))))
        el = run(n)
        close()
        out[label] = (solves * n / el, n, B)
    return {"value": out["all"][0], "unit": UNIT, "cores": cores, "kind": "port", "value_1thread": out["1thread"][0],
            "sample": f"{out['all'][1]} passes over the {out['all'][2]} robots of rank 0's first {a.config} batch, statically split over "
                      f"{cores} native threads (oracle/mt_pool.c); single thread: {out['1thread'][1]} passes over its first {out['1thread'][2]} robots; "
                      f"oracle/ C restatement of NLPClass::step_timing_opti_loop, PRMPCClass::body_theta_mpc and EiQuadProg at -O3 "
                      f"-march=native (the reference itself needs Eigen, absent here, and compiles the body MPC only at horizon 4)"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    run, solves, close, B = cpu_pool(a, cores)
    steps = a.steps
    W = min(max(a.warmup, 1), 5)
    run(W)
    times = [run(1) for _ in range(steps)]
    close()
    tot = sum(times)
    v = solves * steps / tot
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
            "warmup": W, "ms_per_step": 1e3 * tot / steps, "higher_is_better": True, "scaling": plan(a, 1)["scaling"],
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(a, max(1, a.gpus)),   # the own arm's config at this N
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"each step = one pass over the {B}-robot {a.config} batch of one GPU at N = 1, statically split over {cores} "
                                       f"native threads (oracle/mt_pool.c; oracle/ C port at -O3 -march=native; host CPU only, the GPU count does not apply)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Polls NVML (SM clock, power, clock-event reasons) every few ms from a thread while the
    timed region runs; only samples taken between start() and stop() are kept."""
    REASONS = {8: "hw_slowdown", 64: "hw_thermal_slowdown", 32: "sw_thermal_slowdown", 4: "sw_power_cap"}

    def __init__(self, index, period=0.002):
        self.index, self.samples, self.run, self.t, self.h = index, [], False, None, None
        self.period = period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    def _poll(self):
        nv = self.nv
        while self.run:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.h is None:
            return
        self.run = True
        self.t = threading.Thread(target=self._poll, daemon=True)
        self.t.start()

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "note": "NVML unavailable"}
        self.run = False
        self.t.join()
        sm = [x[0] for x in self.samples]
        reasons = set()
        for _, _, rs in self.samples:
            for bit, nm in self.REASONS.items():
                if rs & bit:
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(self.max_sm),
                "power_w_max": max((x[1] for x in self.samples), default=None), "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------- GPU arm
# DRAM bytes (read + write) of the body-MPC tick's kernels per call, from `ncu --set full` captures of this bench's
# body kernel at the batch sizes below (profile constants, not measured in the run): see the named file
TRAFFIC_PROFILE = {}          # filled from profiles/traffic.json when present: {"<nh>:<B>": bytes}
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "traffic.json")


def dbg(msg):
    if os.environ.get("BENCH_DEBUG"):
        print(f"[bench rank {os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


def run_b200(a):
    import torch
    import quadrupedal_loco_b200 as q

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # every rank's host side (pinned buffers, feeder threads) lives on the NUMA node of its own GPU
    from quadrupedal_loco_b200 import sharding as _sh
    numa_note = _sh.pin_to_gpu_numa_node(local) if world > 1 else "single rank: not bound"
    dist = None
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own log lines (version banner, INFO when the caller asks for
        # them) go to stderr; the debug LEVEL is whatever the environment sets and is never touched here
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    p = plan(a, world)
    nh, K, W = a.nh, a.steps, max(a.warmup, 3)
    lo, hi = shard_range(p["B_global"], rank, world) if p["name"] == "cfg3" else (0, p["B_global"] // world)
    B = hi - lo
    per = -(-p["B_global"] // world)
    cfg = {"lamda": p["body_lamda"], "step": {"lamda": p["step_lamda"]}}
    mpc = q.Go1Mpc(local, cfg)
    lib, hh = mpc.lib, mpc.h
    stream = torch.cuda.Stream(device=dev)           # lane 0; every lane is a torch stream handed to the C ABI by its raw pointer
    in_s, out_s, dg_s, tk_s = q.body_in_stride(nh), q.body_out_stride(nh), q.body_diag_stride(nh), q.body_tick_in_stride(nh)

    # ---- inputs: nrot distinct batches, footprint > 2.2x L2 ----
    per_batch = B * (in_s + q.STEP_STATE + q.STEP_IN) * 8
    L = a.lanes or int(min(16, max(2, 2 ** int(round(np.log2(65536 / max(B, 1)))))))
    nrot = int(min(64, max(2, np.ceil(2.2 * L2_BYTES / per_batch))))
    nrot = -(-nrot // L) * L             # a multiple of the lane count: a slot's buffers are only ever used on one lane
    body, stick, sst, sinp = make_inputs(a, rank, world, nrot, mpc.step_default_state())
    rec = np.stack([q.pack_body_inputs(nh, d["tick"], d["tx"], d["theta"], d["bstate"], d["x_warm"], d["refs"]) for d in body])   # [nrot, B, in_s]
    rec_h = torch.from_numpy(rec).pin_memory()
    in_d = rec_h.to(dev)
    out_d = torch.zeros(nrot, B, out_s, dtype=torch.float64, device=dev)
    diag_d = torch.zeros(nrot, B, dg_s, dtype=torch.int32, device=dev)
    soa = lambda x: np.ascontiguousarray(np.stack(x).transpose(0, 2, 1))              # [nrot, F, B]
    st_h = torch.from_numpy(soa(sst)); si_h = torch.from_numpy(soa(sinp)).pin_memory()
    tk_h = torch.from_numpy(np.stack(stick).astype(np.int32)).pin_memory()
    st_d, si_d, tk_d = st_h.to(dev), si_h.to(dev), tk_h.to(dev)
    so_d = torch.zeros(nrot, q.STEP_OUT, B, dtype=torch.float64, device=dev)
    sd_d = torch.zeros(nrot, q.STEP_DIAG, B, dtype=torch.int32, device=dev)

    lanes = [stream] + [torch.cuda.Stream(device=dev) for _ in range(L - 1)]
    lane_ptr = [x.cuda_stream for x in lanes]
    st_w = torch.zeros(L, q.STEP_STATE, B, dtype=torch.float64, device=dev)          # planner state after the tick, per lane
    torch.cuda.synchronize()
    P_in = [in_d[r].data_ptr() for r in range(nrot)]; P_out = [out_d[r].data_ptr() for r in range(nrot)]
    P_dg = [diag_d[r].data_ptr() for r in range(nrot)]
    P_tk = [tk_d[r].data_ptr() for r in range(nrot)]; P_st = [st_d[r].data_ptr() for r in range(nrot)]
    P_si = [si_d[r].data_ptr() for r in range(nrot)]; P_so = [so_d[r].data_ptr() for r in range(nrot)]
    P_sd = [sd_d[r].data_ptr() for r in range(nrot)]; P_sw = [st_w[k].data_ptr() for k in range(L)]

    def chk(rc, what="call"):
        if rc != 0:
            raise RuntimeError(f"{what} failed ({rc}): {lib.go1mpc_last_error(hh).decode()}")

    def launch_sqp(i, lane=0):
        r = i % nrot       # out of place: the pristine state stays put, the lane's working copy receives the new state
        chk(lib.go1mpc_step_timing_step_batch(hh, 3, B, P_tk[r], P_st[r], P_sw[lane], P_si[r], P_so[r], P_sd[r], lane_ptr[lane]), "step_timing")

    def launch_body(i, lane=0):
        r = i % nrot
        chk(lib.go1mpc_body_mpc_step_batch(hh, nh, B, P_in[r], P_out[r], P_dg[r], lane_ptr[lane]), "body_mpc")

    def step(i, lane=0):
        """one robot batch through both ticks, planner first (step-timing -> body-MPC chain) on one stream"""
        launch_sqp(i, lane)
        launch_body(i, lane)

    def fork():
        for k in range(1, L):
            chk(lib.go1mpc_stream_wait(hh, lane_ptr[k], lane_ptr[0]))

    def join():
        for k in range(1, L):
            chk(lib.go1mpc_stream_wait(hh, lane_ptr[0], lane_ptr[k]))

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- setup pass (untimed): every slot once on every lane it will use -> workspaces exist, diag records filled ----
    for i in range(max(nrot, L)):
        step(i, i % L)
    torch.cuda.synchronize()
    diag_all = diag_d.cpu().numpy()
    body_status = diag_all[:, :, 0]
    flops_per_batch = diag_all[:, :, 9].astype(np.float64).sum(axis=1)          # [nrot]
    # the solve kernel's share: instances that entered the active-set loop (at least one add), their flops minus the
    # factorisation / inverse / unconstrained minimiser (n^3/3 + n^3/3 + 2 n^2), which the setup kernel does
    n_ = 2 * nh
    setup_flops = float(n_ ** 3 // 3 + n_ ** 3 // 3 + 2 * n_ * n_)
    entered = diag_all[:, :, 3] > 0
    solve_flops_per_batch = ((diag_all[:, :, 9].astype(np.float64) - setup_flops) * entered).sum(axis=1)
    mean_iters = diag_all[:, :, 2:6].reshape(-1, 4).mean(axis=0)
    mean_l2a = diag_all[:, :, 8].mean()
    sdiag = sd_d.cpu().numpy()
    sqp_solves = sdiag[:, 4, :].astype(np.int64).sum(axis=1)                     # [nrot] QPs the SQP really solved
    sqp_status = sdiag[:, 5::11, :][:, :3, :]
    # algorithmic flops of the planner tick (SURVEY.md 8d closed form for the (4,1,24) QP: 0.15 k + 0.35 k per
    # outer pass; front-end 0.6 k per SQP iteration)
    sqp_outer = sdiag[:, 7::11, :][:, :3, :].astype(np.float64)
    sqp_flops_per_batch = (150.0 * (sqp_status >= 0) + 350.0 * sqp_outer * (sqp_status >= 0) + 600.0).sum(axis=(1, 2))
    solves_per_step = B + float(np.mean(sqp_solves))
    dfma_gflops = mpc.measure_dfma_peak(300)

    dbg("setup pass done")
    # ---- device-resident leg: the K-step schedule, captured once, launched once inside the timed region ----
    def enqueue_steps(n, first=0):
        fork()
        for i in range(first, first + n):
            step(i, i % L)
        join()

    graph = ctypes.c_void_p()
    l_cap0 = mpc.launch_count
    if not a.no_graph:
        chk(lib.go1mpc_graph_capture_begin(hh, lane_ptr[0]), "graph_capture_begin")
        enqueue_steps(K)
        chk(lib.go1mpc_graph_capture_end(hh, lane_ptr[0], ctypes.byref(graph)), "graph_capture_end")
    launches_per_K = mpc.launch_count - l_cap0
    if graph:
        # one untimed launch of the graph: uploads it to the device and brings every rank's GPU to its working clocks (the
        # W warm-up steps of an idle GPU are a fraction of a millisecond); the timed launch below then starts warm on all ranks
        chk(lib.go1mpc_graph_launch(hh, graph, lane_ptr[0]), "graph_launch")
        torch.cuda.synchronize()
    enqueue_steps(W)                                   # warm-up: W untimed steps
    torch.cuda.synchronize()
    # NVML polling takes driver locks shared by every process of the box: 2 ms period on one GPU, 10 ms when 8 ranks poll
    clocks = ClockSampler(local, period=0.002 if world == 1 else 0.010)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    clocks.start()
    l0 = mpc.launch_count
    t_host = time.perf_counter()
    e0.record(stream)
    if a.no_graph:
        enqueue_steps(K)
    else:
        chk(lib.go1mpc_graph_launch(hh, graph, lane_ptr[0]), "graph_launch")
    e1.record(stream)
    t_host = time.perf_counter() - t_host
    e1.synchronize()
    torch.cuda.synchronize()
    barrier()
    if a.dump_outputs:
        # what the caller of both ticks receives from the last timed step (K - 1: slot r on lane ln), taken before the legs
        # below overwrite those buffers: body output records and diagnostics [B, stride], planner Vec38, state after the tick
        # and diagnostics (transposed from the planner's field-major layout to [B, fields])
        r, ln = (K - 1) % nrot, (K - 1) % L
        dump_outputs(a.dump_outputs, {"body_out": out_d[r].cpu().numpy(), "body_diag": diag_d[r].cpu().numpy(),
                                      "step_out": so_d[r].cpu().numpy().T, "step_state": st_w[ln].cpu().numpy().T,
                                      "step_diag": sd_d[r].cpu().numpy().T},
                     lo if p["name"] == "cfg3" else rank * B, DUMP_BYTES // world, "" if world == 1 else f"_rank{rank}")
    launches = (mpc.launch_count - l0) if a.no_graph else launches_per_K
    total_ms = e0.elapsed_time(e1)
    solves_timed = float(sum(B + sqp_solves[i % nrot] for i in range(K)))
    if graph:
        lib.go1mpc_graph_destroy(hh, graph)

    dbg("device leg done")
    # ---- lone single-batch timings (CUDA events around exactly one call / one step, nothing else in flight) ----
    n_lat = max(100, a.latency_samples)

    def timed(fn, n):
        out = np.empty(n)
        ea = [torch.cuda.Event(enable_timing=True) for _ in range(2 * n)]
        for i in range(n):
            ea[2 * i].record(stream); fn(i); ea[2 * i + 1].record(stream)
            ea[2 * i + 1].synchronize()
        for i in range(n):
            out[i] = ea[2 * i].elapsed_time(ea[2 * i + 1])
        return out
    lat_ms = timed(step, n_lat)
    body_ms = timed(launch_body, min(n_lat, 300))
    sqp_ms = timed(launch_sqp, min(n_lat, 300))
    # per-kernel durations of the body tick's three launches (CUDA events recorded by the library around each launch of a lone
    # call): the solve kernel is the dominant kernel of the step
    phase_ms = None
    try:
        mpc.body_phase_timing(True)
        acc = np.zeros(3); n_ph = min(n_lat, 100)
        for i in range(n_ph):
            launch_body(i)
            acc += np.array(mpc.body_phase_ms())
        mpc.body_phase_timing(False)
        if acc[1] > 0:
            phase_ms = acc / n_ph
            solve_fl = float(np.mean(solve_flops_per_batch[np.arange(n_ph) % nrot]))
    except Exception:
        phase_ms = None
    clk = clocks.stop()
    handed_over = mpc.body_handover_total(); guard_trips = mpc.body_guard_trips()

    t = torch.tensor([total_ms, solves_timed], dtype=torch.float64, device=dev)
    ms_by_rank = [total_ms / K]
    if dist:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        ms_by_rank = [float(x[0].item()) / K for x in allt]
        # clocks of every rank's GPU: lowest median SM clock, union of the throttle reasons
        names = sorted(ClockSampler.REASONS.values())
        c = torch.tensor([clk["sm_mhz"] or 0.0] + [1.0 if nm in clk["reasons"] else 0.0 for nm in names], dtype=torch.float64, device=dev)
        cmin = c.clone(); dist.all_reduce(cmin, op=dist.ReduceOp.MIN)
        cmax = c.clone(); dist.all_reduce(cmax, op=dist.ReduceOp.MAX)
        clk = dict(clk, sm_mhz=float(cmin[0].item()), reasons=[nm for i, nm in enumerate(names) if cmax[1 + i].item() > 0],
                   scope="all ranks: lowest median SM clock, union of reasons")
        total_ms_max, solves_all = float(tmax[0].item()), float(tsum[1].item())
    else:
        total_ms_max, solves_all = total_ms, solves_timed
    value = solves_all / (total_ms_max * 1e-3)

    # ---- e2e leg: go1mpc_control_tick_host_async with pinned host buffers (+ the gather to rank 0 for N > 1) ----
    e2e = None
    if not a.no_e2e:
        from quadrupedal_loco_b200 import sharding
        Ke = K
        Le = min(L, 4)
        CD = q.COMPACT_DOUBLES
        tx_np, xw_np, tick_np = q.split_body_record(nh, rec.reshape(nrot * B, in_s))
        R_tx = torch.from_numpy(tx_np).to(dev).view(nrot, B, 28)
        R_out = torch.zeros(nrot, B, out_s, dtype=torch.float64, device=dev)
        R_out[:, :, 18:18 + 2 * nh] = torch.from_numpy(xw_np).to(dev).view(nrot, B, 2 * nh)
        ti_h = torch.from_numpy(tick_np).view(nrot, B, tk_s).pin_memory()
        # N > 1: the result rows of every rank go to rank 0 once per batch.  Default: each rank's tick stores its rows straight into
        # rank 0's buffer over NVLink peer memory and raises a flag there (sharding.PeerGather); --gather nccl: torch.distributed.gather
        pg, gathers, gather_kind = None, [None] * Le, None
        if dist:
            if a.gather == "peer":
                try:
                    pg = sharding.PeerGather(lib, local, per, CD, Le)
                    gather_kind = "peer"
                except Exception as ex:
                    dbg(f"peer gather unavailable ({ex}); falling back to the NCCL gather")
                    pg = None
            if pg is None:
                gathers = [sharding.ResultGather(per, CD, torch.float64, dev) for _ in range(Le)]
                gather_kind = "nccl"
        comp_d = [g.local if g else torch.zeros(per, CD, dtype=torch.float64, device=dev) for g in gathers]
        comp_ptr = [pg.dest(ln) if pg else comp_d[ln].data_ptr() for ln in range(Le)]
        host_rows = world * per if rank == 0 else 0
        comp_h = [torch.zeros(max(host_rows, 1), CD, dtype=torch.float64).pin_memory() for _ in range(Le)]
        ticks = []
        for i in range(nrot * Le):
            r, ln = i % nrot, (i // nrot) % Le
            t_ = q.ControlTick()
            t_.n_sqp, t_.nh = 3, nh
            t_.tick = tk_h[r].data_ptr(); t_.step_in = si_h[r].data_ptr(); t_.body_tick_in = ti_h[r].data_ptr()
            t_.step_state_src_d = P_st[r]; t_.step_state_d = P_sw[ln]
            t_.tx_d = R_tx[r].data_ptr(); t_.body_out_d = R_out[r].data_ptr()
            t_.compact_d = comp_ptr[ln]
            t_.compact = comp_h[ln].data_ptr() if not dist else None
            t_.step_in_rows = SENSOR_ROWS       # the 10 sensor rows; external heights / terrain rows are zero in this workload
            ticks.append(t_)
        torch.cuda.synchronize()

        def e2e_enqueue(i):
            r, ln = i % nrot, i % Le
            if pg and not a.e2e_no_gather:
                pg.acquire(ln, lane_ptr[ln])                           # peers: device-side wait until rank 0 released the slot
            chk(lib.go1mpc_control_tick_host_async(hh, B, ctypes.byref(ticks[r + nrot * ln]), lane_ptr[ln]), "control_tick_host_async")
            if dist and not a.e2e_no_gather:
                if pg:
                    pg.publish(ln, lane_ptr[ln])                       # the tick's pack kernel wrote the rows into rank 0's block
                    if rank == 0:
                        pg.wait_all(ln, lane_ptr[ln])
                        with torch.cuda.stream(lanes[ln]):
                            comp_h[ln].view(world, per, CD).copy_(pg.block(ln), non_blocking=True)
                        pg.release(ln, lane_ptr[ln])
                else:
                    with torch.cuda.stream(lanes[ln]):
                        allrows = gathers[ln].gather()                     # NCCL, once per batch
                        if rank == 0:
                            comp_h[ln].view(world, per, CD).copy_(allrows, non_blocking=True)

        # One CUDA graph per batch slot: the slot's whole call sequence (H2D copies from its pinned buffers, both ticks, the result
        # rows to rank 0, rank 0's D2H) is captured ONCE through the ABI's capture helpers and replayed with one launch per step --
        # the per-step host cost of ~15 CUDA calls is what bounds small per-GPU batches (0.14 ms per 4096-robot step on one GPU).
        # Not with the NCCL gather (a collective enqueued by torch.distributed is not captured here).
        e2e_graphs = None
        torch.cuda.synchronize()
        barrier()                                              # the ranks enter the gather protocol together
        if not a.e2e_no_graph and (pg is not None or not dist) and nrot % Le == 0:
            e2e_enqueue(0); torch.cuda.synchronize()           # workspaces of every stream exist before anything is captured
            for ln in range(Le):
                e2e_enqueue(ln)
            torch.cuda.synchronize()
            e2e_graphs = []
            for r in range(nrot):
                ge = ctypes.c_void_p()
                chk(lib.go1mpc_graph_capture_begin(hh, lane_ptr[r % Le]), "graph_capture_begin")
                e2e_enqueue(r)
                chk(lib.go1mpc_graph_capture_end(hh, lane_ptr[r % Le], ctypes.byref(ge)), "graph_capture_end")
                e2e_graphs.append(ge)

        def e2e_step(i):
            if e2e_graphs is not None:
                r = i % nrot
                chk(lib.go1mpc_graph_launch(hh, e2e_graphs[r], lane_ptr[r % Le]), "graph_launch")
            else:
                e2e_enqueue(i)

        go = threading.Barrier(2)
        done = threading.Event()
        n_feed = [0]

        def feeder():
            torch.cuda.set_device(local)
            while True:
                go.wait()
                if n_feed[0] <= 0:
                    return
                for i in range(n_feed[0]):
                    e2e_step(i)
                done.set()
        th = threading.Thread(target=feeder, daemon=True)
        th.start()                                        # created and parked BEFORE the timed region

        def run_e2e(n):
            n_feed[0] = n
            done.clear()
            fork()
            go.wait()                                     # releases the feeder
            done.wait()
            join()
        dbg("e2e buffers ready")
        run_e2e(max(3, Le))
        torch.cuda.synchronize()
        dbg("e2e warm-up done")
        barrier()
        l1 = mpc.launch_count
        ee0 = torch.cuda.Event(enable_timing=True); ee1 = torch.cuda.Event(enable_timing=True)
        t_wall = time.perf_counter()
        ee0.record(stream)
        run_e2e(Ke)
        ee1.record(stream)
        ee1.synchronize()
        t_wall = time.perf_counter() - t_wall
        torch.cuda.synchronize()
        barrier()
        e2e_launches = int(mpc.launch_count - l1)
        dbg("e2e timed run done")
        # the rows rank 0 holds for the last step on lane 0 against the device-resident leg's results of that slot
        i_chk = ((Ke - 1) // Le) * Le
        r_chk = i_chk % nrot
        want = np.zeros((B, CD))
        so = so_d[r_chk].cpu().numpy(); bo = out_d[r_chk].cpu().numpy(); sdg = sdiag[r_chk]; bdg = diag_all[r_chk]
        want[:, 0:3] = so[0:3].T; want[:, 3:7] = bo[:, 0:4]; want[:, 7] = so[29]; want[:, 8] = so[31]; want[:, 9] = so[35]
        ns = sdg[4]
        last = np.where(ns > 0, sdg[5 + 11 * np.clip(ns - 1, 0, 4), np.arange(B)], -1)
        want[:, 10] = last; want[:, 11] = bdg[:, 0]
        if rank == 0 and not (dist and a.e2e_no_gather):
            got = comp_h[0].numpy()[:B]
            assert np.array_equal(got, want, equal_nan=True), "e2e result rows differ from the device-resident leg"
        gather_ms = None
        if dist and not a.e2e_no_gather:
            # digest check of the gather: sum over all ranks of the local rows == sum of what rank 0 received
            loc = torch.from_numpy(want).to(dev).nansum().reshape(1)
            dist.all_reduce(loc, op=dist.ReduceOp.SUM)
            if rank == 0:
                tot = float(comp_h[0].view(world, per, CD).nansum().item())
                assert abs(tot - float(loc.item())) <= 1e-6 * max(1.0, abs(tot)), "gathered rows do not add up to the ranks' rows"
            # the gather alone: the rows of one batch to rank 0 + rank 0's read-back, CUDA events, 50 repetitions
            g0 = torch.cuda.Event(enable_timing=True); g1 = torch.cuda.Event(enable_timing=True)
            rows_src = torch.zeros(per, CD, dtype=torch.float64, device=dev)
            dst_view = torch.as_tensor(sharding._DevView(pg.dest(0), (per, CD)), device=dev) if pg else None
            barrier()
            with torch.cuda.stream(lanes[0]):
                g0.record(lanes[0])
                for _ in range(50):
                    if pg:
                        pg.acquire(0, lane_ptr[0])
                        dst_view.copy_(rows_src)                       # a device kernel storing the rows into rank 0's block
                        pg.publish(0, lane_ptr[0])
                        if rank == 0:
                            pg.wait_all(0, lane_ptr[0])
                            comp_h[0].view(world, per, CD).copy_(pg.block(0), non_blocking=True)
                            pg.release(0, lane_ptr[0])
                    else:
                        allrows = gathers[0].gather()
                        if rank == 0:
                            comp_h[0].view(world, per, CD).copy_(allrows, non_blocking=True)
                g1.record(lanes[0])
            g1.synchronize()
            gt = torch.tensor([g0.elapsed_time(g1) / 50], dtype=torch.float64, device=dev)
            dist.all_reduce(gt, op=dist.ReduceOp.MAX)
            gather_ms = float(gt.item())
        dbg("e2e checks done")
        # host-to-host latency of ONE batch through the same entry (wall clock on the calling thread, nothing else in flight)
        lat_e2e = []
        n_le = max(100, a.latency_samples) if B <= 16384 else max(100, a.latency_samples // 4)
        for i in range(8 + n_le):
            t0 = time.perf_counter()
            e2e_step(i * Le)                      # lane 0
            lanes[0].synchronize()
            if i >= 8:
                lat_e2e.append(1e3 * (time.perf_counter() - t0))
        lat_t = torch.tensor([np.percentile(lat_e2e, 50), np.percentile(lat_e2e, 99), max(lat_e2e)], dtype=torch.float64, device=dev)
        if dist:
            dist.all_reduce(lat_t, op=dist.ReduceOp.MAX)
        n_feed[0] = 0
        go.wait()
        th.join()
        if pg is not None:
            assert pg.status() == 0, "a device-side wait of the peer gather timed out"

        se = float(sum(B + sqp_solves[i % nrot] for i in range(Ke)))
        te = torch.tensor([ee0.elapsed_time(ee1), se], dtype=torch.float64, device=dev)
        if dist:
            tm = te.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            tsu = te.clone(); dist.all_reduce(tsu, op=dist.ReduceOp.SUM)
            te_ms, se_all = float(tm[0].item()), float(tsu[1].item())
        else:
            te_ms, se_all = float(te[0].item()), se
        h2d = B * (tk_s * 8 + SENSOR_ROWS * 8 + 4)
        d2h = (world * per if dist else B) * CD * 8
        e2e = {"value": se_all / (te_ms * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "bytes_def": "per rank H2D: tick (4 B) + the 10 planner sensor inputs (estimated CoM state, foot locations; flat ground) + (9 + 9 nh) body-tick doubles per robot; D2H: 12-double result rows"
                            + (" of ALL ranks, on rank 0 only (the other ranks ship theirs over NVLink)" if dist else ""),
               "gather_ms": gather_ms,
               "gather": gather_kind,
               "gather_def": ((("every rank's tick stores its [%d][12] result rows straight into rank 0's buffer over NVLink peer memory and "
                                "raises a flag there (csrc/peer_gather.cu: no collective, no rendezvous); rank 0 waits for the flags on the "
                                "device, then D2H of the gathered block" if gather_kind == "peer" else
                                "NCCL gather (torch.distributed.gather) of every rank's [%d][12] result rows into rank 0's device buffer + rank "
                                "0's D2H of the gathered block") % per)
                              + ", once per batch inside the timed region; gather_ms = that exchange alone (50 repetitions, CUDA events, "
                                "max over ranks)") if dist else None,
               "latency_ms": {"p50": float(lat_t[0].item()), "p99": float(lat_t[1].item()), "max": float(lat_t[2].item()),
                              "samples": n_le,
                              "what": f"one {B}-robot batch host to host through the same entry (enqueue, synchronize its stream), wall clock "
                                      f"on the calling thread, max over ranks"},
               "steps": Ke, "ms_per_step": te_ms / Ke, "wall_ms_per_step": 1e3 * t_wall / Ke, "launches": e2e_launches,
               "api": "go1mpc_control_tick_host_async (pinned host buffers; per call on one of %d caller streams: H2D of the tick's arguments, "
                      "planner tick, body tick on the device-resident records, 12-double result row per robot%s); planner state, body step "
                      "table and previous body output record resident on the device; %s; one feeder thread, created and parked before the "
                      "timed region; CUDA events recorded before its release and after the last stream has joined"
                      % (Le, "; the rows go to rank 0 once per batch (see gather_def), then rank 0's D2H" if dist else ", D2H of the rows",
                         "every batch slot's call sequence captured once (go1mpc_graph_capture_*) and replayed with ONE graph launch per step, "
                         "copies included" if e2e_graphs is not None else "every call enqueued from the host each step"),
               "graph_replay": e2e_graphs is not None}

    if rank == 0:
        kern_ms = float(np.mean(body_ms))
        fl = float(np.mean(flops_per_batch[np.arange(len(body_ms)) % nrot]))
        call_tf = fl / (kern_ms * 1e-3) / 1e12
        peak_tf = dfma_gflops / 1e3
        # dominant kernel = tri_solve_kernel when the three-launch path ran (phase events); else the whole call
        if phase_ms is not None:
            dom_name, dom_ms, dom_fl = f"tri_solve_kernel<{nh}, 4> (active-set iteration of the body-inclination MPC tick)", float(phase_ms[1]), solve_fl
            dom_def = (f"mean duration of the solve kernel's launch inside a LONE body-tick call on {B} robots (CUDA events recorded by the library "
                       f"around that launch on the launching stream, go1mpc_body_phase_timing; {min(n_lat, 100)} calls)")
            dom_fdef = ("algorithmic flops of the dense reference algorithm's active-set loop (SURVEY.md 8d formula without its n^3/3 + n^3/3 + 2 n^2 "
                        "set-up terms, n = 2 nh, m = 12 nh) of the instances that enter the loop, counted per problem on the device; the kernel "
                        "exploits G = blockdiag(H, H) and executes fewer")
        else:
            dom_name, dom_ms, dom_fl = "body-inclination MPC tick (go1mpc_body_mpc_step_batch)", kern_ms, fl
            dom_def = f"mean duration of a LONE call on {B} robots (CUDA events around exactly one call on the launching stream)"
            dom_fdef = "algorithmic flops of the dense reference algorithm along each problem's path (SURVEY.md 8d formula), counted per problem on the device"
        achieved_tf = dom_fl / (dom_ms * 1e-3) / 1e12
        io_bytes = B * ((in_s + out_s) * 8 + dg_s * 4)
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]; hbm_src = "measured (MEASURED_PEAKS.json)"
        except Exception:
            hbm_peak = 6650.0; hbm_src = "fallback of B200_PROFILING.md"
        try:
            traffic = json.load(open(TRAFFIC_FILE)).get(f"{nh}:{B}")
        except Exception:
            traffic = None
        traffic_call = None
        if isinstance(traffic, dict):
            traffic_call = traffic.get("body_tick_call")
            traffic = traffic.get("tri_solve_kernel") if phase_ms is not None else traffic_call
        sqp_fl = float(np.mean(sqp_flops_per_batch))
        sqp_k_ms = float(np.mean(sqp_ms))
        step_flops = fl + sqp_fl
        ms_per_step = total_ms_max / K
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": p["scaling"], "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(a, world),
            "solves_per_step_per_gpu": solves_per_step, "robot_ticks_per_s": world * B * K / (total_ms_max * 1e-3),
            "timed_region": ("one CUDA-graph launch of the K-step schedule (captured, uploaded and launched once untimed before the W warm-up steps)" if not a.no_graph
                             else "host enqueue of the K steps") + f", steps dealt over {L} streams, {nrot} distinct input batches",
            "host_ms_in_timed_region": 1e3 * t_host,
            "latency_ms": {"p50": float(np.percentile(lat_ms, 50)), "p99": float(np.percentile(lat_ms, 99)),
                           "max": float(lat_ms.max()), "samples": int(len(lat_ms)),
                           "what": f"one {B}-robot batch through both ticks on one stream (inputs resident in HBM), CUDA events"},
            "kernels_ms": {"body_tick_alone": kern_ms, "step_timing_tick_alone": sqp_k_ms, "step_both_alone": float(np.mean(lat_ms))},
            "body_path": {"mode": os.environ.get("GO1MPC_BODY_MODE", "auto"), "handed_to_combined_kernel": int(handed_over),
                          "guard_trips": int(guard_trips), "not_converged_frac": float((body_status != 0).mean())},
            "roofline": {"bound": "fp64", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak_tf if peak_tf else None,
                         "frac_step": step_flops / (ms_per_step * 1e-3) / 1e12 / peak_tf if peak_tf else None,
                         "frac_step_def": "algorithmic flops of BOTH ticks of one step / the timed ms_per_step / peak",
                         "traffic": traffic,
                         "traffic_source": "profile constant: dram__bytes_read.sum + dram__bytes_write.sum of that kernel for one launch, "
                                           "ncu --set full, profiles/traffic.json (null: no capture at this batch size)",
                         "kernel": dom_name,
                         "kernel_ms": dom_ms,
                         "kernel_ms_def": dom_def,
                         "flops_per_launch": dom_fl, "flops_per_solve": dom_fl / B,
                         "flops_def": dom_fdef,
                         "body_tick_call": {"what": "the whole body-inclination MPC tick (go1mpc_body_mpc_step_batch: setup, solve, merge and the "
                                                    "empty list-mode launch), LONE call, CUDA events around exactly one call",
                                            "kernel_ms": kern_ms, "flops_per_launch": fl, "flops_per_solve": fl / B, "traffic": traffic_call,
                                            "achieved": call_tf, "frac": call_tf / peak_tf if peak_tf else None,
                                            "phases_ms": ({"tri_setup_kernel": float(phase_ms[0]), "tri_solve_kernel": float(phase_ms[1]),
                                                           "tri_merge_kernel": float(phase_ms[2])} if phase_ms is not None else None)},
                         "peak_source": "measured live on this GPU: register-resident DFMA loop (go1mpc_measure_dfma_peak); "
                                        "MEASURED_PEAKS.json has no FP64 figure",
                         "hbm": {"achieved": io_bytes / (kern_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "peak_source": hbm_src, "bytes_per_launch": io_bytes},
                         "other_kernels": {"step_timing_tick": {
                             "kernel_ms": sqp_k_ms, "flops_per_launch": sqp_fl,
                             "achieved": sqp_fl / (sqp_k_ms * 1e-3) / 1e12,
                             "frac": sqp_fl / (sqp_k_ms * 1e-3) / 1e12 / peak_tf if peak_tf else None}}},
            "solver": {"body_mean_outer": float(mean_iters[0]), "body_mean_add": float(mean_iters[1]),
                       "body_mean_drop": float(mean_iters[2]), "body_mean_degen": float(mean_iters[3]),
                       "body_mean_l2a": float(mean_l2a), "sqp_solves_per_robot": float(np.mean(sqp_solves)) / B,
                       "sqp_converged_frac": float((sqp_status == 0).mean()), "sqp_infeasible_frac": float((sqp_status == 2).mean())},
            "clocks": clk, "ms_per_step_by_rank": ms_by_rank, "host_numa": numa_note, "gpu_launches": int(launches), "e2e": e2e,
        }
        if world == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(a)
        print(json.dumps(line), flush=True)
    dbg("closing")
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    mpc.close()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
