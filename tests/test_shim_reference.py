"""CPU: the pybind drop-in `hipie_b200.MultiScaleDeformableAttention` against the reference wrapper
(projects/HIPIE/hipie/models/deformable_detr/ops/functions/ms_deform_attn_func.py).  The fixture tests/golden/ref_msda_binding.pt
records the positional argument list the reference's `MSDeformAttnFunction.forward` passes to `ms_deform_attn_forward` and the
output of its `ms_deform_attn_core_pytorch` on the same inputs.  Here the check is the binding: the shim accepts that argument
list, CPU tensors fail the way the reference op does ("Not implemented on the CPU", ops/src/ms_deform_attn.h:38), and the
reference's pure-PyTorch core agrees with the oracle restatement.  The numerical check of the same call chain on CUDA is
tests/test_model_gpu.py::test_pybind_shim_through_reference_style_function."""
import os
import sys

import pytest
import torch
from torch.autograd import Function


def test_reference_wrapper_binds_to_shim(monkeypatch, golden_dir):
    import hipie_b200.MultiScaleDeformableAttention as shim
    g = torch.load(os.path.join(golden_dir, "ref_msda_binding.pt"))
    monkeypatch.setitem(sys.modules, "MultiScaleDeformableAttention", shim)
    import MultiScaleDeformableAttention as MSDA
    assert MSDA is shim
    named = dict(g["inputs"], im2col_step=g["im2col_step"])
    names = list(named)
    seen = {}
    real = shim.ms_deform_attn_forward

    def spy(*args):
        seen["n"] = len(args)
        seen["im2col_step"] = args[-1]
        return real(*args)
    monkeypatch.setattr(shim, "ms_deform_attn_forward", spy)

    class MSDeformAttnFunction(Function):
        """forwards its inputs in the order the reference wrapper does (recorded in the fixture)"""
        @staticmethod
        def forward(ctx, *inputs):
            by_name = dict(zip(names, inputs))
            return MSDA.ms_deform_attn_forward(*[by_name[n] for n in g["call"]])

    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        MSDeformAttnFunction.apply(*named.values())
    assert seen == {"n": 6, "im2col_step": 64}
    # and the reference's own pure-PyTorch core agrees with the oracle restatement used everywhere else
    from hipie_oracle.msda import ms_deform_attn_core
    x = g["inputs"]
    assert torch.allclose(g["core"], ms_deform_attn_core(x["value"], x["shapes"], x["sampling_loc"], x["attn_weight"]))
