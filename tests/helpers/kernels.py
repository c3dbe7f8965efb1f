"""Which interval kernels a call launched, as the CUDA profiler (CUPTI) reports them.

A handle's reported variant is what construction chose; a launcher may still decline a shape and let the next one in
the chain run.  Tests that must know which instantiation produced their numbers ask the profiler instead."""
import re

_KERNEL_RE = re.compile(r"(?<![A-Za-z0-9_])(bilinear_(?:persistent|dmma|octet|generic|product)_kernel|tdb_(?:dmma_|exp_)?kernel)(<[^>(]*>)?")


def norm(name):
    """A demangled instantiation name without whitespace, bool template arguments spelled false / true."""
    return re.sub(r"\s+", "", name).replace("(bool)0", "false").replace("(bool)1", "true")


def interval_kernels(fn):
    """Run fn() under the CUDA profiler; the set of interval-kernel instantiations it launched (normalised names)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    found = set()
    for e in prof.events():
        m = _KERNEL_RE.search(e.name)
        if m:
            found.add(norm(m.group(0)))
    return found
