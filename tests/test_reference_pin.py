"""Pins against outputs of the REFERENCE's own kernels.

tests/golden/ref_triton_norms.pt holds what the reference's triton/ops/group_norm.py and
layer_norm.py (unmodified) computed under Triton's interpreter -- see
tests/golden/make_reference_golden.py; the inputs are rebuilt from their seed by
tests/golden/reference_inputs.py and the outputs are sampled.  Rows a4 (GroupNorm / GroupNorm +
SiLU) and a9 (LayerNorm) of SURVEY.md section 8 are therefore pinned to reference-run vectors
(zero-mean cases at the reference's own 1e-2; the large-mean case with the reference's own fp16
arithmetic error added, see _stat_slack):

  * CPU (`-m "not gpu"`): oracle/ops_oracle.py against the reference outputs;
  * GPU (`-m gpu`): the CUDA kernels (fused and two-pass GroupNorm, stand-alone LayerNorm, and
    the LayerNorm folded into a tcgen05 GEMM) through the C ABI against the same outputs.

Tolerance = the reference's own self-test: assert_close(rtol=1e-2, atol=1e-2)
(group_norm.py:499,523; layer_norm.py:435 uses atol=1e-2, rtol=0).  Note the reference round-trips
mean / rstd through fp16 (group_norm.py:405-416), so ITS outputs carry ~1e-2 of error against an
fp32 evaluation; the CUDA path keeps the statistics in fp32 and is compared with that slack.
"""
import math
import os

import pytest
import torch

from golden import reference_inputs as ri
from oracle import ops_oracle as oo

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_triton_norms.pt")
GOLDEN_GEGLU = os.path.join(os.path.dirname(__file__), "golden", "ref_cutlass_geglu.pt")


def _check_inputs(case, *tensors):
    """The rebuilt inputs are the ones the reference was run on."""
    for got, want in zip(ri.input_check(*tensors), case["input_check"], strict=True):
        assert torch.equal(got, want), "reference_inputs no longer rebuilds the fixture's inputs"


def _fx():
    """The fixture with each case's inputs (x, weight, bias) rebuilt from their seed."""
    fx = torch.load(GOLDEN)
    gn, ln = ri.norm_cases()
    for case, inp in zip(fx["group_norm"] + fx["layer_norm"], gn + ln, strict=True):
        assert case["tag"] == inp["tag"]
        _check_inputs(case, inp["x"], inp["weight"], inp["bias"])
        case.update(x=inp["x"], weight=inp["weight"], bias=inp["bias"])
    return fx


def _at(y, case):
    """The elements (GroupNorm, NCHW flat indices) or rows (LayerNorm) the fixture kept of y."""
    if "idx" in case:
        return y.flatten()[case["idx"].long().to(y.device)]
    return y[case["rows"].long().to(y.device)]


def _close(got, ref, rtol=1e-2, atol=1e-2):
    torch.testing.assert_close(got.float().cpu(), ref.float().cpu(), rtol=rtol, atol=atol)


def _stat_slack(case, key):
    """Extra absolute slack for a reference OUTPUT on inputs with |mean| >> sigma.  The reference's
    channels_last apply kernel works in the INPUT dtype end to end (group_norm.py:295-318: mean,
    rstd, gamma, beta are fp16, `a = rstd * gamma`, `b = beta - a * mean`, `x = a * x + b` all in
    fp16) after storing mean / rstd in fp16 (group_norm.py:405-416).  So its own result is off by
    about |a| * (|mean - mean_fp16| + 2^-10 * |mean|): ~0 for zero-mean data, ~0.15 when the data
    sit at 50 +- 1.  The CUDA path and the oracle compute in fp32; this is the reference's error,
    documented here, not a tolerance the product path needs."""
    n = case["x"].shape[0]
    xf = case["x"].float().reshape(n, case["groups"], -1)
    mean = xf.mean(-1)
    dmean = (mean - case["mean_" + key].float()).abs().max()
    a = case["weight"].float().abs().max() * case["rstd_" + key].float().max()
    return float(a * (dmean + 2.0 ** -10 * mean.abs().max()))


def _with_reference_stats(case, key, silu):
    """The op evaluated in fp32 from the reference's OWN stored (fp16) statistics: isolates the
    arithmetic of the apply step from the statistics round trip."""
    x = case["x"].float()
    n, c = x.shape[:2]
    cpg = c // case["groups"]
    mean = case["mean_" + key].float().repeat_interleave(cpg, 1)[:, :, None, None]
    rstd = case["rstd_" + key].float().repeat_interleave(cpg, 1)[:, :, None, None]
    y = (x - mean) * rstd * case["weight"].float()[None, :, None, None] + case["bias"].float()[None, :, None, None]
    return y * torch.sigmoid(y) if silu else y


def test_fixture_was_produced_by_the_reference_files():
    fx = _fx()
    assert fx["generator"].endswith("make_reference_golden.py")
    assert "triton/ops/group_norm.py" in fx["reference_files"]
    assert len(fx["group_norm"]) >= 4 and len(fx["layer_norm"]) >= 3
    tags = [c["tag"] for c in fx["group_norm"]]
    assert "selftest_2x320x32x32" in tags  # the reference self-test configuration


@pytest.mark.parametrize("silu", [False, True])
def test_ops_oracle_group_norm_matches_reference_triton_outputs(silu):
    key = "silu" if silu else "plain"
    for case in _fx()["group_norm"]:
        got = oo.group_norm(case["x"], case["groups"], case["weight"], case["bias"], case["eps"], silu)
        slack = _stat_slack(case, key)
        _close(_at(got, case), case["y_nhwc_" + key], atol=1e-2 + slack)
        _close(_at(_with_reference_stats(case, key, silu), case), case["y_nhwc_" + key], atol=1e-2 + slack)
        if "y_nchw_" + key in case:
            _close(_at(got, case), case["y_nchw_" + key], atol=1e-2 + slack)
        # the statistics themselves (the reference stores them in fp16)
        n, c = case["x"].shape[:2]
        xf = case["x"].float().reshape(n, case["groups"], -1)
        _close(xf.mean(-1), case["mean_" + key], rtol=1e-3, atol=2e-3)  # fp16 storage of the mean
        _close(1.0 / torch.sqrt(xf.var(-1, unbiased=False) + case["eps"]), case["rstd_" + key],
               rtol=2e-3, atol=2e-3)


def test_ops_oracle_layer_norm_matches_reference_triton_outputs():
    for case in _fx()["layer_norm"]:
        got = oo.layer_norm(case["x"], case["weight"], case["bias"], case["eps"])
        _close(_at(got, case), case["y"], rtol=0, atol=1e-2)


# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("silu", [False, True])
def test_cuda_group_norm_matches_reference_triton_outputs(silu, fused):
    from sfast_b200 import _lib, ops
    from sfast_b200.ops import Act
    lib = _lib.lib()
    key = "silu" if silu else "plain"
    for case in _fx()["group_norm"]:
        x = case["x"].cuda()
        n, c, h, w = x.shape
        xb = x.permute(0, 2, 3, 1).contiguous()                      # the path's NHWC layout
        yb = torch.zeros_like(xb)
        stats = torch.empty(ops.gn_ws_floats(n, case["groups"]), device="cuda")
        sync = torch.zeros(4, device="cuda", dtype=torch.int32)
        gops = ops.gn_ops("gn", lib, x=Act(xb, n, h, w, c), y=Act(yb, n, h, w, c),
                          gamma=case["weight"].cuda().float(), beta=case["bias"].cuda().float(),
                          stats=stats, groups=case["groups"], eps=case["eps"], silu=silu,
                          dt=torch.float16, sync=sync if fused else None)
        assert len(gops) == (1 if fused else 2)
        for op in gops:
            op.launch(torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        _close(_at(yb.permute(0, 3, 1, 2), case), case["y_nhwc_" + key], atol=1e-2 + _stat_slack(case, key))
        # and tightly against the fp32-statistics oracle (what the reference approximates)
        want = oo.group_norm(case["x"], case["groups"], case["weight"], case["bias"], case["eps"], silu)
        _close(yb.permute(0, 3, 1, 2), want, rtol=4e-3, atol=4e-3)


@pytest.mark.gpu
def test_cuda_layer_norm_and_folded_layer_norm_match_reference_triton_outputs():
    from sfast_b200 import _lib, ops
    lib = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    for case in _fx()["layer_norm"]:
        x = case["x"].cuda()
        rows, c = x.shape
        gamma, beta = case["weight"].cuda().float(), case["bias"].cuda().float()
        # (1) stand-alone kernel
        y = torch.zeros_like(x)
        ops.ln_op("ln", lib, x=x, y=y, rows=rows, c=c, gamma=gamma, beta=beta, eps=case["eps"],
                  dt=torch.float16).launch(st)
        torch.cuda.synchronize()
        _close(_at(y, case), case["y"], rtol=0, atol=1e-2)
        # and the whole output tightly against the fp32 oracle
        _close(y, oo.layer_norm(case["x"], case["weight"], case["bias"], case["eps"]), rtol=4e-3, atol=4e-3)
        # (2) the product path: LayerNorm folded into the consuming tcgen05 GEMM.  Row statistics as
        # the producer epilogue would leave them (sum, sum of squares of the stored fp16 row); the
        # expected result is the REFERENCE LayerNorm output pushed through the same linear in fp32,
        # on the rows the fixture kept.
        torch.manual_seed(1)
        n_out = 320
        w = (torch.randn(n_out, c, device="cuda") / math.sqrt(c)).half()
        b = torch.randn(n_out, device="cuda") * 0.1
        wp, bias, colsum = ops.fold_layer_norm(w, b, gamma, beta, torch.float16)
        xf = x.float()
        stats = torch.stack([xf.sum(-1), (xf * xf).sum(-1)], dim=-1).contiguous()
        out = torch.zeros(rows, n_out, device="cuda", dtype=torch.float16)
        ops.gemm_op("consumer", lib, a=ops.a_matrix(x.data_ptr(), rows, c, c), b=ops.Mat(wp.contiguous()),
                    M=rows, N=n_out, K=c, dt=torch.float16, out=out, ldo=n_out, bias=bias, splits=1,
                    ln=dict(rowstats=stats, colsum=colsum, eps=case["eps"], dim=c)).launch(st)
        torch.cuda.synchronize()
        ref = case["y"].cuda().float() @ w.float().t() + b
        # the reference LN output is itself fp16-rounded: allow its quantisation through the GEMM
        _close(_at(out, case), ref, rtol=1e-2, atol=2e-2)
        # and every row against the fp16-rounded oracle LayerNorm pushed through the same linear
        want = oo.layer_norm(x, gamma, beta, case["eps"]).float() @ w.float().t() + b
        _close(out, want, rtol=1e-2, atol=2e-2)


# ------------------------------------------------------------------------------------------------
# Row a7: Linear + GEGLU pinned against the reference's own CUTLASS kernel run on a B200
# (the reference's csrc/operators/cutlass/cutlass_dual_linear_kernel.cu, compiled from its own
# source by oracle/build_ref.sh); tests/golden/ref_cutlass_geglu.pt holds its outputs -- see
# tests/golden/make_reference_geglu_golden.py.
def _geglu_fx():
    return torch.load(GOLDEN_GEGLU)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("shape", ri.GEGLU_SHAPES)
def test_cuda_geglu_matches_reference_cutlass_kernel(dtype, shape):
    """UNet GEGLU sizes (the reference's benchmark test uses in_features 320 / 640 -> 1280 / 2560,
    tests/operators/test_cutlass_dual_linear.py:59-72) at the reference's tolerance 2e-2: the
    reference kernel's output, the oracle and the tcgen05 GEMM + GEGLU epilogue must agree.  The
    reference accumulates in fp16 / bf16 and uses the tanh GELU under torch's default flags
    (cutlass_dual_linear_kernel.cu:391-393,509-514); the CUDA path accumulates in fp32 with erf."""
    from sfast_b200 import _lib, ops
    case = next(c for c in _geglu_fx()["unet"]
                if c["dtype"] == str(dtype).replace("torch.", "") and tuple(c["shape"]) == shape)
    lib = _lib.lib()
    m, k, inner = shape
    x, w, b = ri.geglu_inputs(dtype, shape)
    _check_inputs(case, x, w, b)
    x, w, b = x.cuda(), w.cuda(), b.cuda()
    ref = case["y"].cuda()
    assert ref.dtype == dtype
    want = oo.linear_geglu(x, w, b)
    wp, bp, _ = ops.pack_geglu(w, b.float(), dtype)
    out = torch.zeros(m, inner, device="cuda", dtype=dtype)
    ops.gemm_op("geglu", lib, a=ops.a_matrix(x.data_ptr(), m, k, k), b=ops.Mat(wp), M=m, N=wp.shape[0],
                K=k, dt=dtype, out=out, ldo=inner, bias=bp, epi=ops.EPI_GEGLU, geglu_n_out=inner,
                splits=1).launch(torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    tol = 2e-2 if dtype == torch.float16 else 6e-2   # the bf16 reference accumulates in bf16
    _close(_at(want, case), ref, rtol=tol, atol=tol)  # oracle  vs reference-run
    _close(_at(out, case), ref, rtol=tol, atol=tol)   # product vs reference-run
    _close(out, want, rtol=1e-2, atol=1e-2)           # product vs oracle (fp32 truth), tighter


@pytest.mark.gpu
@pytest.mark.parametrize("bias", [False, True])
def test_reference_cutlass_kernel_on_its_own_test_configuration(bias):
    """The reference's own small-shape test (tests/operators/test_cutlass_dual_linear.py:42-56,
    n in (4, 16), in / out features in (8, 16)) run against the oracle -- checks the oracle's chunk
    order / GELU against the reference binary's outputs."""
    cases = [c for c in _geglu_fx()["own_config"] if (c["bias"] is not None) == bias]
    assert len(cases) == 8
    for c in cases:
        x, wt = c["x"].cuda(), c["weight"].cuda()
        bs = c["bias"].cuda() if bias else None
        _close(oo.linear_geglu(x, wt, bs), c["y"], rtol=2e-2, atol=2e-2)
