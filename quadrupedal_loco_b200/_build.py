"""In-tree build of libgo1mpc.so (sm_100a only).  nvcc cross-compiles without a GPU."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgo1mpc.so")
SOURCES = ["api.cu", "body_mpc.cu", "body_fast.cu", "body_tri.cu", "body_duo.cu", "body_resident.cu", "qp_dense.cu", "step_timing.cu", "step_sqp.cu", "foot_traj.cu", "leg_kin.cu", "grf_qp.cu", "ref_interp.cu", "rt_chain.cu", "nlp_chain.cu", "filters.cu", "peer_gather.cu", "gait_stack.cu", "servo_stack.cu", "servo_torque.cu", "farm_health.cu"]
# A/B variants that `auto` never chooses (body_split.cu: roll / pitch halves side by side in one warp) are only compiled
# into the library with GO1MPC_BUILD_AB=1 (then GO1MPC_BODY_MODE=split selects it)
AB_SOURCES = ["body_split.cu"]
# per-source extra flags: the thread-per-instance kernels keep the oracle's operation order and
# must not contract a*b+c into FMA
EXTRA = {"step_timing.cu": ["-fmad=false"], "step_sqp.cu": ["-fmad=false"], "foot_traj.cu": ["-fmad=false"], "leg_kin.cu": ["-fmad=false"], "ref_interp.cu": ["-fmad=false"], "rt_chain.cu": ["-fmad=false"], "nlp_chain.cu": ["-fmad=false"], "filters.cu": ["-fmad=false"],
         "servo_stack.cu": ["-fmad=false"], "servo_torque.cu": ["-fmad=false"]}
HEADERS = ["gi_warp.cuh", "grf_math.cuh", "tma.cuh", "powi.cuh", "servo_math.cuh", "kernels.h", os.path.join("..", "..", "include", "go1mpc.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    # host code builds tables that are asserted bit-identical to the reference's (build_body_model, build_aaa_inv_mod):
    # GCC's default -ffp-contract=fast would contract a*b+c on FMA-baseline hosts (aarch64, -march=native)
    "-Xcompiler", "-ffp-contract=off",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libgo1mpc.so cannot be built (there is no CPU fallback)")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + AB_SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile every CUDA source (one object each, in parallel) and link quadrupedal_loco_b200/libgo1mpc.so."""
    if not force and not needs_build():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    extra = os.environ.get("GO1MPC_NVCC_EXTRA", "").split()
    sources = list(SOURCES)
    if os.environ.get("GO1MPC_BUILD_AB") == "1":
        sources += AB_SOURCES
        extra += ["-DGO1MPC_AB_VARIANTS"]
    # the image exports CC/CXX=/opt/gcc/bin/* whose link line picks a static libstdc++;
    # let nvcc use the PATH host compiler instead
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + extra + EXTRA.get(src, []) + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, cwd=CSRC, env=env, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + r.stdout + r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=len(sources)) as ex:
        results = list(ex.map(compile_one, sources))
    if verbose:
        for _, err in results:
            print(err)
    r = subprocess.run([_nvcc(), "-shared", "-o", LIB] + [o for o, _ in results], cwd=CSRC, env=env, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
