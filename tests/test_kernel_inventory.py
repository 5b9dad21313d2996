"""CPU suite: librtiow_cuda.so carries exactly the kernels the host side can launch.

Each instantiation of render_kernel, hitlist_kernel and ray_color_kernel (and their tensor-core twins) is named by one arm of
the scan plan (plan_scan in capi.cu), and for render_kernel by one kind of render launch (rt::Loop) too.  An instantiation no
arm launches is dead code that costs compile time and library size.
"""
import re
import subprocess

LOOPS = ["Frame", "Views", "Aov", "Adaptive"]       # rt::Loop in declaration order: c++filt prints (rt::Loop)0 .. (rt::Loop)3
RENDER_ARMS = {
    "render_kernel<double, false, 256, 2, {}>": "F64: rtiow_render at RTIOW_PRECISION_F64 tests every sphere",
    "render_kernel<float, true, 256, 3, {}>": "Smem: the FP32 filter's table in shared memory, three 256-thread CTAs per SM",
    "render_kernel<float, true, 768, 1, {}>": "Wide: a table too large for 256-thread CTAs, one 768-thread CTA per SM when its lists fit",
    "render_kernel<float, true, 512, 1, {}>": "Wide: the same with 512 threads when the 768-thread lists do not fit",
    "render_kernel<float, false, 256, 4, {}>": "Global: a table too large for shared memory, read from global memory",
    "render_kernel_umma<6, 64, {}>": "Tensor: the tensor-core filter (RT_UMMA_GROUPS, RT_UMMA_CHUNK)",
}
EXPECTED = {arm.format(f"Loop::{loop}"): why for arm, why in RENDER_ARMS.items() for loop in LOOPS} | {
    "hitlist_kernel<double, false, 256>": "F64: rtiow_hitlist_batch at RTIOW_PRECISION_F64",
    "hitlist_kernel<float, true, 256>": "Smem",
    "hitlist_kernel<float, true, 512>": "Wide (the unit kernels always use 512 threads there)",
    "hitlist_kernel<float, false, 256>": "Global",
    "hitlist_kernel_umma<6, 64>": "Tensor",
    "ray_color_kernel<double, false, 256>": "F64: rtiow_ray_color_batch at RTIOW_PRECISION_F64",
    "ray_color_kernel<float, true, 256>": "Smem",
    "ray_color_kernel<float, true, 512>": "Wide (the unit kernels always use 512 threads there)",
    "ray_color_kernel<float, false, 256>": "Global",
    "ray_color_kernel_umma<6, 64>": "Tensor",
}
# the other kernels of a render call: one quantising epilogue for every kind of launch and destination, the AOV epilogue, the
# de-interleave of gathered tile buffers, and the rounds of rtiow_render_adaptive
FRAME_KERNELS = {"finalize_kernel", "finalize_aov_kernel", "deinterleave_kernel", "adapt_first_list_kernel", "adapt_select_kernel",
                 "adapt_compact_kernel"}


def test_kernel_instantiations_are_the_plan_arms(capi):
    syms = subprocess.run(["cuobjdump", "-symbols", str(capi.lib_path())], capture_output=True, text=True, check=True).stdout
    names = subprocess.run(["c++filt"], input=syms, capture_output=True, text=True, check=True).stdout
    found = {re.sub(r"\(rt::Loop\)(\d)", lambda m: f"Loop::{LOOPS[int(m.group(1))]}", n)
             for n in re.findall(r"rt::((?:render|hitlist|ray_color)_kernel(?:_umma)?<[^>]*>)", names)}
    assert found == set(EXPECTED), f"unexpected: {sorted(found - set(EXPECTED))}, missing: {sorted(set(EXPECTED) - found)}"
    frame = set(re.findall(r"STO_ENTRY\s+rt::((?:finalize|deinterleave|adapt)\w*)\(", names))
    assert frame == FRAME_KERNELS, f"unexpected: {sorted(frame - FRAME_KERNELS)}, missing: {sorted(FRAME_KERNELS - frame)}"
