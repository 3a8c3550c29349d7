"""Room beside a resident scoring CTA (DESIGN.md section 4).

In the streaming evaluator a batch's row normalise and list merge run while a neighbouring stream's scoring kernel
holds one CTA per SM.  At cfg 2 (B = 512, C = 21,841, D = 1,024) one CTA of the scoring kernel, one of the normalise
and two of the merge must fit on one SM together in shared memory, and the scoring CTA, a normalise and a merge CTA
in registers; otherwise the small CTAs of a step wait for an SM without a scoring CTA.  The limits are the device's
and the footprints are the built kernels' as the library launches them, both read at run time.
"""
import ctypes

import pytest
import torch

from hgrnet_b200 import ops

pytestmark = pytest.mark.gpu

SMEM_UNIT = 128   # shared memory is granted to a CTA in 128-byte units
REG_UNIT = 8      # registers per thread are granted in steps of 8 (256 per warp)

# CUdevice_attribute
MAX_SMEM_PER_SM = 81
MAX_REGS_PER_SM = 82
RESERVED_SMEM_PER_BLOCK = 111


def _device_limits():
    torch.cuda.init()
    cu = ctypes.CDLL("libcuda.so.1")
    dev = ctypes.c_int()
    assert cu.cuDeviceGet(ctypes.byref(dev), torch.cuda.current_device()) == 0
    out = {}
    for name, attr in (("smem_per_sm", MAX_SMEM_PER_SM), ("regs_per_sm", MAX_REGS_PER_SM),
                       ("reserved_smem_per_block", RESERVED_SMEM_PER_BLOCK)):
        v = ctypes.c_int()
        assert cu.cuDeviceGetAttribute(ctypes.byref(v), attr, dev) == 0
        out[name] = v.value
    return out


def _smem(fp, reserved):
    need = fp["static_smem"] + fp["dynamic_smem"]
    return -(-need // SMEM_UNIT) * SMEM_UNIT + reserved


def _regs(fp):
    return -(-fp["registers"] // REG_UNIT) * REG_UNIT * fp["threads"]


@pytest.mark.parametrize("x_dtype", [torch.bfloat16, torch.float32])
def test_normalise_and_two_merges_fit_beside_a_scoring_cta_at_cfg2(x_dtype):
    lim = _device_limits()
    fp = ops.score_topk_footprint(512, 21841, 1024, 20, x_dtype=x_dtype)
    smem = sum(_smem(f, lim["reserved_smem_per_block"]) for f in (fp["score"], fp["normalize"], fp["merge"], fp["merge"]))
    regs = sum(_regs(f) for f in (fp["score"], fp["normalize"], fp["merge"]))
    assert smem <= lim["smem_per_sm"], (smem, lim, fp)
    assert regs <= lim["regs_per_sm"], (regs, lim, fp)
