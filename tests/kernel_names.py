"""Which instantiations of the rollout family (k_rollouts, k_rollouts_wide, k_opt_risk) the library holds, and which ones a call launched.

`built_instantiations` reads the template instantiations from the host stubs of libmpcmmd.so (`nm -C`).  `launched` runs a call under
torch.profiler with CUDA activities and returns the names of the kernels it ran, graph-launched ones included.  Both give names in one
form, e.g. "k_rollouts<1, true, 0, 0>", so that a test can state the instantiation its launch must reach and check it."""
import re
import subprocess

FAMILY = re.compile(r"\b(k_rollouts_wide|k_rollouts|k_opt_risk)<([^<>()]*)>")


def normalize(name):
    """the rollout-family instantiation named in a demangled symbol or kernel name ("k_rollouts<1, true, 0, 0>"), or None"""
    m = FAMILY.search(name)
    if not m:
        return None
    return f"{m.group(1)}<{', '.join(a.strip() for a in m.group(2).split(','))}>"


def built_instantiations(lib_path):
    """every rollout-family instantiation whose host stub is in the library"""
    out = subprocess.run(["nm", "-C", lib_path], check=True, capture_output=True, text=True).stdout
    return {n for n in (normalize(line) for line in out.splitlines()) if n}


def launched(fn):
    """(fn's result, the set of kernel names the GPU ran during fn).  Fails when the profiler saw no CUDA kernel at all: a test that
    states which kernel its launch reaches must not pass because nothing was recorded."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith("Memcpy")
             and not e.name.startswith("Memset")}
    assert names, "torch.profiler recorded no CUDA kernel for the call"
    return out, names


def family(names):
    """the rollout-family instantiations among kernel names"""
    return {n for n in (normalize(k) for k in names) if n}
