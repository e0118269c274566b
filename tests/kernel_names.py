"""Which instantiations of a kernel family the library holds, and which ones a call launched.

Two families: "rollout" (k_rollouts, k_rollouts_wide, k_opt_risk) and "inner" (the reduced-set inner CEM of mmd_opt: k_inner_cem_fast,
k_inner_cem_lat, k_inner_cem and k_inner_cem_big).  `built_instantiations` reads the template instantiations from the host stubs of
libmpcmmd.so (`nm -C`).  `launched` runs a call under torch.profiler with CUDA activities and returns the names of the kernels it ran,
graph-launched ones included.  Both give names in one form, e.g. "k_rollouts<1, true, 0, 0>", so that a test can state the instantiation
its launch must reach and check it."""
import re
import subprocess

FAMILIES = {
    "rollout": re.compile(r"\b(k_rollouts_wide|k_rollouts|k_opt_risk)<([^<>()]*)>"),
    "inner": re.compile(r"\b(k_inner_cem_fast|k_inner_cem_lat|k_inner_cem_big|k_inner_cem)<([^<>()]*)>"),
}


def normalize(name, which="rollout"):
    """the instantiation of family `which` named in a demangled symbol or kernel name ("k_rollouts<1, true, 0, 0>"), or None"""
    m = FAMILIES[which].search(name)
    if not m:
        return None
    return f"{m.group(1)}<{', '.join(a.strip() for a in m.group(2).split(','))}>"


def built_instantiations(lib_path, which="rollout"):
    """every instantiation of family `which` whose host stub is in the library"""
    out = subprocess.run(["nm", "-C", lib_path], check=True, capture_output=True, text=True).stdout
    return {n for n in (normalize(line, which) for line in out.splitlines()) if n}


def _profiled(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith("Memcpy")
             and not e.name.startswith("Memset")}
    return out, names


def launched(fn):
    """(fn's result, the set of kernel names the GPU ran during fn).  fn must give the same result when called again (a stage or a solve
    of fixed inputs).  torch.profiler occasionally returns a session with no records at all when one process has opened many of them, so
    an empty session runs fn once more under a new one; the call fails when that one is empty too: a test that states which kernel its
    launch reaches must not pass because nothing was recorded."""
    out, names = _profiled(fn)
    if not names:
        out, names = _profiled(fn)
    assert names, "torch.profiler recorded no CUDA kernel for the call"
    return out, names


def family(names, which="rollout"):
    """the instantiations of family `which` among kernel names"""
    return {n for n in (normalize(k, which) for k in names) if n}
