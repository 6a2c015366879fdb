"""Build recipe for libml4ca_b200.so (nvcc, sm_100a only, in-tree).

`python -m ml4ca_b200.build` or `__graft_entry__.build()`.  The shared library is written next to
this file so that it travels to the GPU box with the repository snapshot.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libml4ca_b200.so")
STAMP = os.path.join(HERE, ".libml4ca_b200.stamp")

# (source, extra defines, object suffix)
SOURCES = [("common.cu", [], ""), ("env_step.cu", [], ""), ("pinv_pid.cu", [], ""), ("qp_alloc.cu", [], ""), ("policy.cu", [], ""), ("gae.cu", [], ""), ("ppo_update.cu", [], ""), ("ppo_update_tc.cu", [], ""), ("ppo_update_generic.cu", [], ""), ("peer_comm.cu", [], ""), ("ros_adapter.cu", [], ""), ("eval_metrics.cu", [], ""), ("observer.cu", [], ""), ("refmodel.cu", [], "")] + \
          [("env_step_inst.cu", ["-DML4CA_STEP_UNIT=%d" % u], "_%d" % u) for u in range(5)]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _digest():
    h = hashlib.sha256()
    files = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))) + ["../../include/ml4ca_b200.h"]
    for f in files:
        path = os.path.join(CSRC, f)
        if os.path.isfile(path):
            h.update(f.encode())
            with open(path, "rb") as fh:
                h.update(fh.read())
    h.update(repr((NVCC_FLAGS, SOURCES)).encode())
    return h.hexdigest()


def build(force=False, verbose=False, extra_flags=(), out=None):
    """Compile every CUDA source into libml4ca_b200.so.  Returns the library path.
    extra_flags/out build an experimental variant next to the default library (tuning only)."""
    global LIB, STAMP
    if out is not None:
        LIB = os.path.join(HERE, out)
        STAMP = LIB + ".stamp"
        force = True
    if not force and _up_to_date(_digest()):
        return LIB      # nothing to write: a read-only tree that was built beforehand loads as it is
    # one builder at a time: under torchrun every rank may get here at once and would write the same .o / .so / stamp files
    import fcntl
    with open(os.path.join(HERE, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose, extra_flags, out)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _up_to_date(digest):
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as fh:
        return fh.read().strip() == digest


def _build_locked(force, verbose, extra_flags, out):
    global LIB, STAMP
    digest = _digest()
    if not force and _up_to_date(digest):
        return LIB
    objs = []
    log = []

    def compile_one(item):
        src, defines, suffix = item
        tag = "" if out is None else "_" + os.path.splitext(out)[0]
        obj = os.path.join(CSRC, src.replace(".cu", suffix + tag + ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + list(extra_flags) + defines + ["-c", os.path.join(CSRC, src), "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, "$ " + " ".join(cmd) + "\n" + res.stdout + res.stderr, res.returncode

    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=min(os.cpu_count() or 4, len(SOURCES))) as pool:
        results = list(pool.map(compile_one, SOURCES))
    for src, obj, text, rc in results:
        log.append(text)
        if rc != 0:
            sys.stderr.write("\n".join(log)[-6000:])
            raise RuntimeError("nvcc failed on %s" % src)
        objs.append(obj)
    # link under a temporary name and rename: a caller that found the stamp current without the lock (build() above) may be
    # loading LIB while a forced rebuild runs, and must see the old or the new library, never a partly written one
    tmp = "%s.tmp%d.so" % (os.path.splitext(LIB)[0], os.getpid())     # still matched by the *.so ignore rule
    cmd = [_nvcc(), "-shared", "-o", tmp] + objs + ["-lcudart"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log.append("$ " + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if res.returncode != 0:
        if os.path.exists(tmp):
            os.remove(tmp)
        sys.stderr.write("\n".join(log)[-6000:])
        raise RuntimeError("link failed")
    os.replace(tmp, LIB)
    with open(os.path.join(HERE, "build.log"), "w") as fh:
        fh.write("\n".join(log))
    with open(STAMP, "w") as fh:
        fh.write(digest)
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
