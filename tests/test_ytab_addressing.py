"""The y-table traversal addresses its per-lane table through one 32-bit shared-window address, set once per thread by the
caller, instead of a generic pointer into dynamic shared memory.  Through the generic pointer every table store of the fill and
every table load of an interior visit rebuilt the window base (S2UR SR_CgaCtaId, UMOV, UIADD3, ULEA): 20 of its reads in each
y-table kernel, 4 of the visit's issue slots.  Without a GPU: the SASS of every y-table function reads SR_CgaCtaId at most as
often as its non-y-table sibling, plus once for each of its two y-table traversal instantiations."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
YT_INSTANTIATIONS = 2                # traverse<false, CNT, false, AX, true> for AX = true and false


def _window_base_reads():
    obj = os.path.join(ROOT, "mirror_maze_b200", "build", "render_kernel.o")
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not (os.path.exists(obj) and os.path.exists(tool)):
        pytest.skip("needs the built render_kernel.o and cuobjdump")
    sass = subprocess.run([tool, "-sass", obj], capture_output=True, text=True, check=True).stdout
    counts, name = {}, None
    for line in sass.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
            counts[name] = 0
        elif name and "SR_CgaCtaId" in line:
            counts[name] += 1
    return counts


# y-table kernel (mangled name part) -> its non-y-table sibling: same body, same template arguments, YT = false
SIBLINGS = [
    (r"17trace_ytab_kernelI(Lb[01]ELb[01]ELi\d+E)E", r"12trace_kernelI\1E"),
    (r"22trace_ytab_wide_kernelI(Lb[01]ELb[01]E)E", r"12trace_kernelI\1Li1024EE"),
    (r"17views_ytab_kernelI(Lb[01]ELb[01]ELi\d+E)E", r"12views_kernelI\1E"),
    (r"22views_ytab_wide_kernelI(Lb[01]ELb[01]E)E", r"17views_wide_kernelI\1E"),
    (r"17trace_tail_kernelI(Lb[01]ELb[01]E)Lb1EE", r"17trace_tail_kernelI\1Lb0EE"),
    (r"17views_tail_kernelI(Lb[01]ELb[01]E)Lb1EE", r"17views_tail_kernelI\1Lb0EE"),
    (r"17probe_rays_kernelILb1EE", r"17probe_rays_kernelILb0EE"),
]


def test_ytab_kernels_set_the_table_window_base_once_per_traversal_at_most():
    counts = _window_base_reads()
    checked = 0
    for pattern, sibling in SIBLINGS:
        for name, n in counts.items():
            m = re.search(pattern, name)
            if not m:
                continue
            twin = name[:m.start()] + m.expand(sibling) + name[m.end():]
            assert twin in counts, (name, twin)
            assert n <= counts[twin] + YT_INSTANTIATIONS, (name, n, counts[twin])
            checked += 1
    # 6 trace_ytab_kernel + 3 wide + 6 views_ytab_kernel + 3 wide + 3 + 3 tail kernels + probe_rays_kernel<true>
    assert checked == 25
