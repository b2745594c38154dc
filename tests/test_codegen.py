"""Code generation of the hot kernels, checked without a GPU on the sm_100a cubins inside csrc/librthx.so.

The tracing kernels sit at their register bounds (64 registers at 4 resident blocks, 80 at 3), so a change that looks unrelated can
push ptxas into spilling inside a ray loop.  Round 2 lost 15 % of the MULTI_BOUNCE rate that way: a pointer dropped from TraceParams
slid the parameter-bank constants by 8 bytes (profiles/r4/r4c_*).  These bounds are the stack frames (= spill space) of the shipped
build; a larger frame must be looked at (and measured) before the bound is raised."""
import re
import shutil
import subprocess

import pytest

# kernel (demangled prefix) -> (registers, largest stack frame in bytes)
BOUNDS = {
    "trace_exchange_sq_kernel<4, false>": (64, 8),                    # cfg1-4: the headline kernel
    "trace_exchange_sq_kernel<4, true>": (64, 24),                    # lock-step MULTI_BOUNCE loop (block_threads < 256)
    "trace_exchange_queue_kernel<4, false, false, false>": (64, 16),  # cfg5: per-warp ray queue, depth 4
    "trace_exchange_queue_kernel<2, false, false, false>": (64, 16),
    "trace_exchange_queue_kernel<4, true, false, false>": (64, 64),   # general faces (bilinear lattices, T-junctions)
    "trace_exchange_queue_kernel<2, false, true, false>": (80, 64),   # MULTI_BOUNCE on the ray queue
    "trace_exchange_queue_kernel<4, true, false, true>": (64, 88),    # generic locator on the ray queue
    "trace_exchange_kernel<true, false, false>": (64, 40),            # generic locator, lock-step (single-face meshes)
}

# every trace-kernel instance the library compiles (rthx_kernels.cu, k_trace_instances): each is reachable by some trace
TRACE_KERNELS = {
    *(f"trace_exchange_kernel<{h}, {f}, {m}>" for h in ("true", "false") for f in ("true", "false") for m in ("true", "false")),
    "trace_exchange_sq_kernel<4, false>", "trace_exchange_sq_kernel<4, true>",
    *(f"trace_exchange_queue_kernel<{d}, {b}, false, false>" for d in (1, 2, 4) for b in ("false", "true")),
    *(f"trace_exchange_queue_kernel<{d}, {b}, true, false>" for d in (1, 2) for b in ("false", "true")),
    "trace_exchange_queue_kernel<2, true, false, true>", "trace_exchange_queue_kernel<4, true, false, true>",
    "trace_exchange_hash_kernel<true>", "trace_exchange_hash_kernel<false>",
}


def _resource_usage(so):
    out = subprocess.run(["cuobjdump", "--dump-resource-usage", so], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)
    dem = subprocess.run(["c++filt"], input="\n".join(n for n, _, _ in names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {d: (int(r), int(s)) for d, (_, r, s) in zip(dem, names)}


@pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("c++filt") is None, reason="needs cuobjdump and c++filt")
def test_hot_kernels_keep_their_registers_and_stack_frames(cuda_lib, rthx_mod):
    usage = _resource_usage(rthx_mod.build_library())
    for prefix, (regs, stack) in BOUNDS.items():
        hits = [(k, v) for k, v in usage.items() if k.startswith("void rthx::" + prefix) or k.startswith("rthx::" + prefix)]
        assert len(hits) == 1, (prefix, [k for k, _ in hits])
        name, (r, s) = hits[0]
        assert r <= regs, f"{name}: {r} registers (bound {regs}: resident blocks per SM would drop)"
        assert s <= stack, f"{name}: stack frame {s} bytes (bound {stack}): ptxas spills more than the measured build"


@pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("c++filt") is None, reason="needs cuobjdump and c++filt")
def test_library_compiles_exactly_the_selectable_trace_kernels(cuda_lib, rthx_mod):
    usage = _resource_usage(rthx_mod.build_library())
    built = {re.sub(r"^(void )?rthx::", "", k).split("(")[0] for k in usage if "trace_exchange" in k}
    assert len(TRACE_KERNELS) == 24
    assert built == TRACE_KERNELS, (sorted(built - TRACE_KERNELS), sorted(TRACE_KERNELS - built))
