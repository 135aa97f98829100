"""CPU-side build evidence (cuobjdump on the in-tree libdfgpu.so): the kernels that run by default are the instantiations that were
measured — 256-bit loads (LDG.E.ENL2.256), L2 prefetches (CCTL.E.PF2) and one RED per lane pair in the fused pipeline kernel and
the paired group-by kernel; the radix scatter moves its tiles with TMA bulk copies.  (profiles/r2c_sass_excerpt_ldg256_paired_red.txt,
profiles/r2_radix_scatter_tma_sass_excerpt.txt hold the excerpts.)"""
import re
import subprocess

from datafusion_b200 import capi
from harness import cuda_tool


def sass(fn):
    out = subprocess.run([cuda_tool("cuobjdump"), "-sass", "-fun", fn, capi.LIB_PATH], capture_output=True, text=True).stdout
    return [l for l in out.splitlines() if re.match(r"\s+/\*[0-9a-f]{4,5}\*/", l)]


def default_of(path, name):
    m = re.search(rf"constexpr int {name} = (\d+);", open(path).read())
    assert m, name
    return int(m.group(1))


def test_default_pipeline_instantiation_has_wide_loads_prefetches_and_paired_reds():
    import os
    var = default_of(os.path.join(os.path.dirname(capi.LIB_PATH), "csrc", "pipeline.cu"), "kPipeVarDefault")
    assert var == 43
    code = sass(f"_ZN5dfgpu11pipe_kernelILi3ELb0ELi{var}EEEvPKNS_10PipeParamsElPy")          # pipe_kernel<SINK_AGG, false, 43>
    assert len(code) > 5000
    assert sum("ENL2.256" in l for l in code) >= 6 and sum("CCTL.E.PF2" in l for l in code) >= 3
    base = sass("_ZN5dfgpu11pipe_kernelILi3ELb0ELi0EEEvPKNS_10PipeParamsElPy")                # the round-start kernel stays available (DFGPU_PIPE_VAR=0)
    assert len(base) > 5000 and not any("ENL2.256" in l or "CCTL.E.PF2" in l for l in base)


def test_default_group_by_kernel_is_the_paired_one_with_the_wide_bucket_load():
    import os
    mode = default_of(os.path.join(os.path.dirname(capi.LIB_PATH), "csrc", "aggregate.cu"), "kAggPairedDefault")
    assert mode == 4
    code = sass("_ZN5dfgpu22agg_update_pair_kernelILi3ELb1EEEvPKyS2_S2_P10ulonglong2NS_8TableDevEllPKjPjPy")   # agg_update_pair_kernel<3, true>
    assert sum("ENL2.256" in l for l in code) == 3                     # one bucket load per row in flight
    assert sum("REDG.E.ADD.64" in l and "@" not in l.split("REDG")[0][-6:] for l in code) == 6   # two per row in flight: even lanes' rows, odd lanes' rows
    assert sum("SHFL.BFLY" in l for l in code) >= 12


def test_radix_scatter_uses_tma_bulk_copies():
    code = sass("_ZN5dfgpu24radix_scatter_tma_kernelEPKyS1_liPyPNS_8RadixRecE")
    assert any("UBLKCP" in l for l in code) and any("SYNCS" in l for l in code)
