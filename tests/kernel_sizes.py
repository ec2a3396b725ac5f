"""Code size of the kernels in libfo_b200.so, read with cuobjdump (used by the CPU code-size budget tests).

The metric kernels are instruction-issue- and instruction-cache-bound (DESIGN.md sections 5.1 and 6), so shared device
code must not quietly push one of them out of the instruction cache.  ``size_of(*parts)`` is the SASS size in bytes of
the one kernel whose mangled name contains every part, out-of-line helpers included.  ``hot=True`` leaves out the cold
float64 re-rounding of np.round(d, 3) ties (obb_round_mm_f64, sincos_f64_of_f32), which runs for a fraction of a per
cent of the exact distance evaluations.  Skips the calling test when the toolkit has no cuobjdump."""
import functools
import os
import re
import shutil
import subprocess

import pytest


@functools.lru_cache(maxsize=None)
def _tables():
    from torch.utils.cpp_extension import CUDA_HOME
    from frenetix_occlusion_b200 import _lib as L
    # the toolkit that built the library has it, whether or not its bin/ is on PATH
    cuobjdump = shutil.which("cuobjdump") or (CUDA_HOME and shutil.which("cuobjdump", path=os.path.join(CUDA_HOME, "bin")))
    if not cuobjdump:
        return None
    sass = subprocess.run([cuobjdump, "-sass", L.LIB_PATH], capture_output=True, text=True).stdout
    sizes, name = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
        elif name and re.match(r"\s+/\*[0-9a-f]+\*/\s+\S", line):
            sizes[name] = sizes.get(name, 0) + 16
    # cold helpers live in the kernel's text section but not in its hot set
    cold = {}
    elf = subprocess.run([cuobjdump, "-elf", L.LIB_PATH], capture_output=True, text=True).stdout
    for line in elf.splitlines():
        m = re.match(r"\s*0x[0-9a-f]+\s+0x[0-9a-f]+\s+(0x[0-9a-f]+)\s+.*\$(_ZN\S+?)\$(_ZN\S+)", line)
        if m and ("obb_round_mm_f64" in m.group(3) or "sincos_f64_of_f32" in m.group(3)):
            cold[m.group(2)] = cold.get(m.group(2), 0) + int(m.group(1), 16)
    return sizes, cold


def size_of(*parts, hot=False):
    tables = _tables()
    if tables is None:
        pytest.skip("cuobjdump not found (no CUDA toolkit)")
    sizes, cold = tables
    hit = [v - (cold.get(k, 0) if hot else 0) for k, v in sizes.items() if all(p in k for p in parts)]
    assert len(hit) == 1, (parts, sorted(sizes))
    return hit[0]
