"""Generates tests/golden/ref_cutlass_geglu.pt: outputs of the REFERENCE's own CUTLASS GEGLU kernel.

What runs: oracle/_ref/libsfast_ref_geglu.so, the reference's cutlass_dual_linear_kernel.cu compiled
from its own source by oracle/build_ref.sh, as torch.ops.sfast_ref.linear_geglu(x, weight, bias) on
a CUDA device.  Under torch's default flags it accumulates in fp16 / bf16 and uses the tanh GELU
(cutlass_dual_linear_kernel.cu:391-393,509-514).

Cases:
  * "unet": the UNet GEGLU sizes of tests/test_reference_pin.py in fp16 and bf16, inputs from
    reference_inputs.geglu_inputs (not stored; the test rebuilds them), reference_inputs.SAMPLES
    sampled output elements each;
  * "own_config": the reference's own small-shape test (tests/operators/test_cutlass_dual_linear.py:
    42-56: n in (4, 16), in / out features in (8, 16), with and without bias, fp16), inputs and
    outputs stored whole.

Run from the repo root on a GPU machine, after build():
    python tests/golden/make_reference_geglu_golden.py [output path]
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from golden import reference_inputs as ri  # noqa: E402

REF_SO = os.path.join(os.path.dirname(os.path.dirname(HERE)), "oracle", "_ref", "libsfast_ref_geglu.so")


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref_cutlass_geglu.pt")
    torch.ops.load_library(REF_SO)
    ref_op = torch.ops.sfast_ref.linear_geglu
    out = {"generator": "tests/golden/make_reference_geglu_golden.py",
           "reference_files": ["csrc/operators/cutlass/cutlass_dual_linear_kernel.cu"],
           "device": torch.cuda.get_device_name(0), "unet": [], "own_config": []}
    for dtype in (torch.float16, torch.bfloat16):
        for i, shape in enumerate(ri.GEGLU_SHAPES):
            x, w, b = ri.geglu_inputs(dtype, shape)
            y = ref_op(x.cuda(), w.cuda(), b.cuda()).cpu()
            assert y.shape == (shape[0], shape[2]) and y.dtype == dtype
            idx = ri.sample_index(y.numel(), seed=i)
            out["unet"].append({"dtype": str(dtype).replace("torch.", ""), "shape": shape, "idx": idx,
                                "y": y.flatten()[idx.long()], "input_check": ri.input_check(x, w, b)})
            print("unet", dtype, shape, "done", flush=True)
    for bias in (False, True):
        for n in (4, 16):
            for cin in (8, 16):
                for cout in (8, 16):
                    torch.manual_seed(n * 100 + cin * 10 + cout)
                    proj = torch.nn.Linear(cin, 2 * cout, bias=bias).half()
                    x = torch.randn(n, cin).half()
                    wb = proj.bias.detach().cuda() if bias else None
                    y = ref_op(x.cuda(), proj.weight.detach().cuda(), wb).cpu()
                    out["own_config"].append({"x": x, "weight": proj.weight.detach(),
                                              "bias": proj.bias.detach() if bias else None, "y": y})
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
