"""Which interval kernels (and which knot-side kernels) a call launched, as the CUDA profiler (CUPTI) reports them.

A handle's reported variant names the kernel family construction chose, and the launchers run exactly that family.  Which
instantiation of it (template arguments, products, split forms) ran is the profiler's to say."""
import re

_KERNEL_RE = re.compile(r"(?<![A-Za-z0-9_])(bilinear_(?:persistent|dmma|octet|generic|product)_kernel|tdb_(?:dmma_|exp_)?kernel)(<[^>(]*>)?")


def norm(name):
    """A demangled instantiation name without whitespace, bool template arguments spelled false / true."""
    return re.sub(r"\s+", "", name).replace("(bool)0", "false").replace("(bool)1", "true")


def _launched(fn, regex):
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    found = set()
    for e in prof.events():
        m = regex.search(e.name)
        if m:
            found.add(norm(m.group(0)))
    return found


def interval_kernels(fn):
    """Run fn() under the CUDA profiler; the set of interval-kernel instantiations it launched (normalised names)."""
    return _launched(fn, _KERNEL_RE)


# the kernels around the interval kernels: Hessian assembly (K3), objective and gradient (K6) with their reductions,
# knot-objective pairs, knot constraints (K5), derivative integrators (K2), terms with global variables (K8), the
# violation reduction and the Jacobian products
_KNOT_RE = re.compile(r"(?<![A-Za-z0-9_])(hessian_assemble(?:_left)?_kernel|objective_kernel|knot_objective_pairs_kernel"
                      r"|constraint_product_kernel|analytic_product_kernel|analytic_kernel|constraint_kernel|knot_program_kernel"
                      r"|global_grad_kernel|global_hess_kernel|column_sum_kernel|kg_sum_kernel|objective_chunk_kernel"
                      r"|objective_reduce_kernel|violation_kernel|jac_product_kernel|hpp_contract_kernel)(?![A-Za-z0-9_])(<[^>]*>)?")


def knot_kernels(fn):
    """Run fn() under the CUDA profiler; the set of knot-side kernel instantiations it launched (normalised names)."""
    return _launched(fn, _KNOT_RE)
