"""Generates tests/golden/ref_triton_norms.pt: outputs of the REFERENCE's own Triton kernels.

What runs: the unmodified files /root/reference/src/sfast/triton/ops/{group_norm,layer_norm,
activation,utils}.py (+ sfast/utils/copy_func.py), imported from where they lie -- nothing is
copied.  `import sfast` itself is impossible here (src/sfast/__init__.py:22-31 needs the compiled
sfast._C), so the package objects `sfast`, `sfast.triton`, `sfast.triton.ops`, `sfast.utils` are
registered as empty namespace modules whose __path__ points into /root/reference: the four kernel
files then import exactly as in the reference.  There is no GPU in this container, so the
@triton.jit kernels execute under Triton's own interpreter (TRITON_INTERPRET=1, numpy on the CPU):
same kernel source, same launch grids, same host wrappers (`group_norm_forward`,
`group_norm_silu_forward`, `LayerNorm.forward`).  Two harness shims, neither touches reference
code: (1) the script must run under `python -O` so the wrappers' `assert input.device.type ==
'cuda'` (group_norm.py:390) is skipped; (2) Triton 3.6's interpreter looks a kernel up by
`fn.__name__` after re-exec'ing its source, which breaks for the reference's renamed copies
(`copy_func(..., name=f'{kernel.__name__}_{act.__name__}')`, group_norm.py:87-96) -- the lookup
falls back to the single function the source defines.

Cases: reference_inputs.norm_cases() -- the reference self-test configuration (group_norm.py:481-527:
randn(2, 320, 32, 32) fp16, G = 32, randn affine, eps 1e-5, NCHW and channels_last, with and without
SiLU), UNet-shaped extras (1280 channels at 8x8, a large-mean input, an outlier channel), and
LayerNorm on the self-test's data recipe (layer_norm.py:406-438: x = -2.3 + 0.5 randn, rand affine)
at UNet widths.  The inputs are not stored (the test rebuilds them from the same seed); of each
output the fixture keeps the GroupNorm statistics whole, reference_inputs.SAMPLES sampled elements
of each GroupNorm output and 32 sampled rows of each LayerNorm output, which keeps it small.

Run from the repo root (about 5 minutes):   python -O tests/golden/make_reference_golden.py
"""
import importlib
import os
import sys
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from golden import reference_inputs as ri  # noqa: E402

REF_ROWS = 32  # LayerNorm output rows kept per case

REF = "/root/reference/src/sfast"


def _load_reference_kernels():
    if __debug__:
        raise SystemExit("run with `python -O` (the reference wrappers assert a CUDA device)")
    os.environ["TRITON_INTERPRET"] = "1"
    from triton.runtime import interpreter as ti

    def compile_and_exec(self, tree):
        code = compile(tree, filename=self.filename, mode="exec")
        ns = {**self.kwargs}
        g = self.fn.__globals__
        for k, v in vars(ti).items():
            if k not in g:
                g[k] = v
        exec(code, g, ns)
        if self.fn.__name__ in ns:
            return ns[self.fn.__name__]
        fns = [v for v in ns.values()
               if getattr(v, "__code__", None) is not None and v.__code__.co_filename == self.filename]
        assert len(fns) == 1, list(ns)
        return fns[0]

    ti.FunctionRewriter._compile_and_exec = compile_and_exec
    for name, path in (("sfast", REF), ("sfast.triton", REF + "/triton"),
                       ("sfast.triton.ops", REF + "/triton/ops"), ("sfast.utils", REF + "/utils")):
        m = types.ModuleType(name)
        m.__path__ = [path]
        sys.modules[name] = m
    gn = importlib.import_module("sfast.triton.ops.group_norm")
    ln = importlib.import_module("sfast.triton.ops.layer_norm")
    assert gn.__file__.startswith(REF) and ln.__file__.startswith(REF)
    return gn, ln


def main():
    gn, ln = _load_reference_kernels()
    out = {"generator": "tests/golden/make_reference_golden.py",
           "reference_files": ["triton/ops/group_norm.py", "triton/ops/layer_norm.py",
                               "triton/ops/activation.py", "triton/ops/utils.py"],
           "group_norm": [], "layer_norm": []}
    gn_cases, ln_cases = ri.norm_cases()
    for i, inp in enumerate(gn_cases):
        tag, x, w, b = inp["tag"], inp["x"], inp["weight"], inp["bias"]
        idx = ri.sample_index(x.numel(), seed=i).long()
        case = {"tag": tag, "groups": inp["groups"], "eps": inp["eps"], "idx": idx.int(),
                "input_check": ri.input_check(x, w, b)}
        xcl = x.contiguous(memory_format=torch.channels_last)
        for silu, fn in ((False, gn.group_norm_forward), (True, gn.group_norm_silu_forward)):
            key = "silu" if silu else "plain"
            if tag.startswith("selftest"):
                case["y_nchw_" + key] = fn(x, 32, w, b, 1e-5)[0].flatten()[idx]
            y, mean, rstd = fn(xcl, 32, w, b, 1e-5)
            assert y.is_contiguous(memory_format=torch.channels_last)
            # NCHW flat indices into the values of the NHWC kernel
            case["y_nhwc_" + key] = y.contiguous().flatten()[idx]
            case["mean_" + key], case["rstd_" + key] = mean, rstd
        out["group_norm"].append(case)
        print("group_norm", tag, "done", flush=True)

    for i, inp in enumerate(ln_cases):
        x, weight, bias, n = inp["x"], inp["weight"], inp["bias"], inp["x"].shape[1]
        y = ln.LayerNorm.forward(types.SimpleNamespace(save_for_backward=lambda *a: None), x, (n,),
                                 weight, bias, 1e-5)
        rows = ri.sample_index(x.shape[0], seed=100 + i, count=REF_ROWS)
        out["layer_norm"].append({"tag": inp["tag"], "eps": inp["eps"], "rows": rows, "y": y[rows.long()],
                                  "input_check": ri.input_check(x, weight, bias)})
        print("layer_norm", inp["tag"], "done", flush=True)

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_triton_norms.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
