"""ctypes access to the CPU oracle (oracle/liboracle.so) and, when present, to the
reference build (oracle/_ref/*.so).  Test infrastructure: nothing in the product
package imports this module."""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORC_DIR = os.path.join(ROOT, "oracle")
dp = ctypes.POINTER(ctypes.c_double)
ip = ctypes.POINTER(ctypes.c_int)


def P(a):
    return a.ctypes.data_as(dp)


def PI(a):
    return a.ctypes.data_as(ip)


class BodyCfg(ctypes.Structure):
    _fields_ = [("nh", ctypes.c_int), ("dt_mpc", ctypes.c_double), ("dt_slow", ctypes.c_double),
                ("tstep", ctypes.c_double), ("height_offset_time", ctypes.c_double), ("g", ctypes.c_double),
                ("mass", ctypes.c_double), ("j_ini", ctypes.c_double), ("foot_length", ctypes.c_double),
                ("foot_width", ctypes.c_double), ("theta_lim", ctypes.c_double), ("torque_lim", ctypes.c_double),
                ("Rtheta", ctypes.c_double), ("alphatheta", ctypes.c_double), ("beltatheta", ctypes.c_double),
                ("gama_zmp", ctypes.c_double), ("lamda", ctypes.c_double * 4)]


class StepCfg(ctypes.Structure):
    _fields_ = [(n, ctypes.c_double) for n in (
        "dt Wn ggg t_min t_max footx_max footx_min footx_vmax footx_vmin footy_vmax footy_vmin comax_max comax_min "
        "comay_max comay_min aax aay aaxv aayv bbx bby rr1 rr2 half_hip_width foot_width").split()] + [
        ("lamda", ctypes.c_double * 4), ("hcom", ctypes.c_double), ("n_sqp", ctypes.c_int), ("ext_height", ctypes.c_int)]


class StepDiag(ctypes.Structure):
    _fields_ = [("periond_i", ctypes.c_int), ("k_yu", ctypes.c_int), ("bjxx", ctypes.c_int), ("bjx1", ctypes.c_int),
                ("n_solved", ctypes.c_int), ("status", ctypes.c_int * 8), ("nactive", ctypes.c_int * 8),
                ("iters", (ctypes.c_int * 4) * 8), ("active", (ctypes.c_int * 25) * 8), ("x", (ctypes.c_double * 4) * 8)]


STEP_STATE, STEP_IN, STEP_OUT = 202, 20, 38


def build_oracle(fast=False):
    """liboracle.so: -O2 -ffp-contract=off (the checker), built in oracle/ when missing or older than its
    sources.  fast=True: liboracle_fast.so, the same sources at -O3 -march=native for the CPU-baseline
    timing, always built afresh on the machine that times it (-march=native code may not run elsewhere)
    and into a new temporary directory (the tree may be read-only there); the caller removes it."""
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    if fast:
        tmp = tempfile.mkdtemp(prefix="go1mpc_oracle_")
        so = os.path.join(tmp, "liboracle_fast.so")
        try:
            subprocess.run(["make", "-s", "-C", ORC_DIR, f"FAST_SO={so}", so], check=True, env=env, capture_output=True)
        except BaseException:
            shutil.rmtree(tmp, ignore_errors=True)
            raise
        return so
    so = os.path.join(ORC_DIR, "liboracle.so")
    srcs = [os.path.join(ORC_DIR, f) for f in os.listdir(ORC_DIR) if f.endswith((".c", ".h"))]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["make", "-s", "-C", ORC_DIR, "liboracle.so"], check=True, env=env, capture_output=True)
    return so


def ref_path(name):
    p = os.path.join(ORC_DIR, "_ref", name)
    return p if os.path.exists(p) else None


class Oracle:
    def __init__(self, fast=False):
        so = build_oracle(fast)
        self.lib = ctypes.CDLL(so)
        if fast:
            shutil.rmtree(os.path.dirname(so))      # the loaded library stays mapped

    def qp_solve(self, n, p, m, G, g0, CE, ce0, CI, ci0, x0=None):
        """Column-major flat inputs for ONE problem.  Returns dict."""
        x = np.zeros(n) if x0 is None else np.array(x0, dtype=float)
        cost = np.zeros(1); act = np.zeros(m + p + 1, np.int32); na = np.zeros(1, np.int32); it = np.zeros(4, np.int32)
        z = np.zeros(1)
        st = self.lib.orc_qp_solve(n, p, m, P(np.ascontiguousarray(G, dtype=float)), P(np.ascontiguousarray(g0, dtype=float)),
                                   P(np.ascontiguousarray(CE, dtype=float)) if p else P(z),
                                   P(np.ascontiguousarray(ce0, dtype=float)) if p else P(z),
                                   P(np.ascontiguousarray(CI, dtype=float)) if m else P(z),
                                   P(np.ascontiguousarray(ci0, dtype=float)) if m else P(z),
                                   P(x), P(cost), PI(act), PI(na), PI(it))
        return dict(status=st, x=x, cost=cost[0], active=act[:na[0]].copy(), nactive=int(na[0]), iters=it)

    def qp_solve_batch(self, n, p, m, d, x0=None):
        B = d["G"].shape[0]
        xs = np.zeros((B, n)); cost = np.zeros(B); status = np.zeros(B, np.int32)
        nact = np.zeros(B, np.int32); iters = np.zeros((B, 4), np.int32); active = np.zeros((B, m + p), np.int32)
        for b in range(B):
            r = self.qp_solve(n, p, m, d["G"][b], d["g0"][b], d["CE"][b], d["ce0"][b], d["CI"][b], d["ci0"][b],
                              None if x0 is None else x0[b])
            xs[b] = r["x"]; cost[b] = r["cost"]; status[b] = r["status"]; nact[b] = r["nactive"]
            iters[b] = r["iters"]; active[b, :r["nactive"]] = r["active"]
        return dict(x=xs, cost=cost, status=status, nactive=nact, iters=iters, active=active)

    def body_cfg(self, nh, **over):
        c = BodyCfg()
        self.lib.orc_body_cfg_default(ctypes.byref(c), nh)
        for k, v in over.items():
            if k == "lamda":
                for i in range(4):
                    c.lamda[i] = v[i]
            else:
                setattr(c, k, v)
        return c

    def body_step_batch(self, cfg, tick, tx, theta, bstate, refs, out14, x):
        """In/out arrays as in orc_body_step_batch; returns diagnostics."""
        B = len(tick); nh = cfg.nh
        tick = np.ascontiguousarray(tick, np.int32)
        act = np.zeros((B, 12 * nh), np.int32); na = np.zeros(B, np.int32); it = np.zeros((B, 4), np.int32)
        st = np.zeros(B, np.int32)
        refs = np.ascontiguousarray(refs.reshape(B, 9 * nh))
        self.lib.orc_body_step_batch(ctypes.byref(cfg), B, PI(tick), P(tx), P(theta), P(bstate), P(refs), P(out14), P(x),
                                     PI(act), PI(na), PI(it), PI(st))
        return dict(active=act, nactive=na, iters=it, status=st)

    # ---- step-location / step-timing SQP ----
    def step_cfg(self, n_sqp=3, **over):
        c = StepCfg()
        self.lib.orc_step_cfg_default(ctypes.byref(c))
        c.n_sqp = n_sqp
        for k, v in over.items():
            if k == "lamda":
                for i in range(4):
                    c.lamda[i] = v[i]
            else:
                setattr(c, k, v)
        return c

    def step_default_state(self, cfg, steplength=0.075, stepwidth=0.2535, stepheight=0.0, tstep=0.7):
        s = np.zeros(STEP_STATE)
        self.lib.orc_step_state_default.argtypes = [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_double] * 4
        self.lib.orc_step_state_default(P(s), ctypes.byref(cfg), steplength, stepwidth, stepheight, tstep)
        return s

    def step_tick_batch(self, cfg, tick, states, ins):
        """Instance-major arrays: states [B,202] (updated in place), ins [B,20].  Returns out [B,38] and
        diagnostics in the GPU diag layout [B,60]."""
        B = len(tick)
        out = np.zeros((B, STEP_OUT)); diag = np.zeros((B, 60), np.int32)
        for b in range(B):
            dg = StepDiag()
            self.lib.orc_step_timing_tick(ctypes.byref(cfg), int(tick[b]), P(states[b]), P(np.ascontiguousarray(ins[b])),
                                          P(out[b]), ctypes.byref(dg))
            diag[b, 0:5] = [dg.periond_i, dg.k_yu, dg.bjxx, dg.bjx1, dg.n_solved]
            for q in range(5):
                o = 5 + 11 * q
                if q < dg.n_solved:
                    st = dg.status[q]
                    diag[b, o] = st; diag[b, o + 1] = 0 if st == 1 else dg.nactive[q]
                    diag[b, o + 2:o + 6] = list(dg.iters[q])
                    na = 0 if st == 1 else dg.nactive[q]
                    diag[b, o + 6:o + 11] = [dg.active[q][k] if k < na else -99 for k in range(5)]
                else:
                    diag[b, o] = -1
        return out, diag

    # ---- leg kinematics (instance-major arrays) ----
    def leg_fk(self, q, leg, bp=None, br=None):
        B = len(leg); pos = np.zeros((B, 3)); J = np.zeros((B, 9))
        for b in range(B):
            if bp is None:
                self.lib.orc_leg_fk(P(np.ascontiguousarray(q[b])), int(leg[b]), P(pos[b]), P(J[b]))
            else:
                self.lib.orc_leg_fk_g(P(np.ascontiguousarray(bp[b])), P(np.ascontiguousarray(br[b])), P(np.ascontiguousarray(q[b])),
                                      int(leg[b]), P(pos[b]), P(J[b]))
        return pos, J

    def leg_ik(self, pdes, qini, leg, bp=None, br=None):
        B = len(leg); q = np.zeros((B, 3)); J = np.zeros((B, 9)); it = np.zeros(B, np.int32)
        for b in range(B):
            if bp is None:
                it[b] = self.lib.orc_leg_ik(P(np.ascontiguousarray(pdes[b])), P(np.ascontiguousarray(qini[b])), int(leg[b]), P(q[b]), P(J[b]))
            else:
                it[b] = self.lib.orc_leg_ik_g(P(np.ascontiguousarray(bp[b])), P(np.ascontiguousarray(br[b])), P(np.ascontiguousarray(pdes[b])),
                                              P(np.ascontiguousarray(qini[b])), int(leg[b]), P(q[b]), P(J[b]))
        return q, J, it

    # ---- swing-foot trajectory ----
    def foot_default_state(self, sw0=0.12675):
        f = np.zeros(32)
        self.lib.orc_foot_state_default.argtypes = [ctypes.c_void_p, ctypes.c_double]
        self.lib.orc_foot_state_default(P(f), sw0)
        return f

    def foot_tick_batch(self, cfg, tick, states_after, bjxx, foot, sw0=0.12675, lift=0.03):
        """states_after [B,202] (after the step tick), bjxx [B], foot [B,32] updated in place -> out18 [B,18], right_support [B]"""
        self.lib.orc_foot_traj_tick.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                                ctypes.c_double, ctypes.c_double, ctypes.c_void_p]
        B = len(tick); out = np.zeros((B, 18)); rs = np.zeros(B, np.int32)
        for b in range(B):
            rs[b] = self.lib.orc_foot_traj_tick(ctypes.byref(cfg), int(tick[b]), P(np.ascontiguousarray(states_after[b])), int(bjxx[b]),
                                                P(foot[b]), sw0, lift, P(out[b]))
        return out, rs
