"""The forced-cooperative test libraries (ddp-generator_b200/lib_coop/, built with -DILQG_FORCE_COOP=1) really hold the
warp-cooperative backward pass and the default libraries do not, so that tests/test_gpu_variants.py compares two different
kernels.  Read from the device code with cuobjdump; no GPU needed."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "ddp-generator_b200")


def _cuobjdump():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not found")
    return exe


def _kernels(lib):
    path = os.path.join(PKG, lib)
    assert os.path.exists(path), f"{path} not built (build() in __graft_entry__.py builds it)"
    out = subprocess.run([_cuobjdump(), "-symbols", path], check=True, capture_output=True, text=True).stdout
    return {k for k in ("k_backpass_warp", "k_backpass_split", "k_backpass") if any(k + "I" in line for line in out.splitlines())}


@pytest.mark.parametrize("problem", ["car", "carhx", "pend", "brachi_hli"])
@pytest.mark.parametrize("ddp", [0, 1])
def test_coop_build_holds_the_cooperative_backward_pass(problem, ddp):
    assert _kernels(f"lib_coop/libilqg_b200_{problem}_ddp{ddp}.so") == {"k_backpass_warp"}


def test_default_build_does_not():
    assert _kernels("lib/libilqg_b200_car_ddp0.so") == {"k_backpass_split", "k_backpass"}
    assert _kernels("lib/libilqg_b200_carhx_ddp0.so") == {"k_backpass"}
    assert _kernels("lib/libilqg_b200_quad_ddp0.so") == {"k_backpass_warp"}
