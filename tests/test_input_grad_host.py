"""CPU: the C-ABI of the network-input gradient (csrc/input_grad.cu) -- declared, exported, plannable without a GPU, and compiled for
sm_100a without local-memory spills."""
import os
import re

import pytest

from pytorch3dunet_b200 import _lib

NEW = ["b200_input_dgrad_partials_count", "b200_input_dgrad_conv3", "b200_gn_bwd_apply_ncdhw_f32", "b200_pointwise_dgrad_f32"]
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "pytorch3dunet_b200", "csrc")


def test_input_grad_entry_points_declared_and_exported():
    protos = _lib.parse_header()
    L = _lib.lib()
    for name in NEW:
        assert name in protos, name
        assert hasattr(L, "_" + name), name


def test_input_dgrad_partials_count_without_gpu():
    L = _lib.lib()
    # MMA path (C_in 1, C_out 8/16/32): one partial per (H x W tile of 8 x 32, chunk of D); the chunk is shortened until >= 512 blocks
    assert L.query("b200_input_dgrad_partials_count", 2, 128, 128, 128, 1, 16) == 16 * 4 * 4
    assert L.query("b200_input_dgrad_partials_count", 2, 19, 23, 17, 1, 8) == 3 * 1 * 5
    # CUDA-core path: one partial per 256 voxels
    assert L.query("b200_input_dgrad_partials_count", 1, 33, 18, 10, 3, 16) == (33 * 18 * 10 + 255) // 256
    assert L.query("b200_input_dgrad_partials_count", 1, 8, 8, 8, 1, 64) == 2


@pytest.mark.parametrize("build", ["build", "build_f16"])
def test_input_grad_kernels_do_not_spill(build):
    log = os.path.join(CSRC, build, "input_grad.ptxas.log")
    if not os.path.exists(log):
        pytest.skip(f"{log} not built")
    text = open(log).read()
    kernels = re.findall(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", text)
    assert len(kernels) >= 6, text
    spills = {k: (st, sl) for k, _, st, sl in kernels if st != "0" or sl != "0"}
    assert not spills, spills
