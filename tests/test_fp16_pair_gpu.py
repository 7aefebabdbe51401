"""GPU: the fp16-pair forward GEMM (dppo_tc_linear_forward format 1; tc3_gemm_kernel<BIAS_TANH, F16>) that the MLP entry points
run for the layers whose input is a tanh output: float64 accuracy over the input range a tanh produces, the per-row weight
scales, non-finite weights, device row counts, and a training step against the FFMA path."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import ppo_oracle as O

F16 = 1
TC_TOL = 3e-5            # the bound tests/test_kernels_gpu.py holds the 3xTF32 forward to
SHAPES = [(4096, 256, 256), (4096, 512, 256), (5000, 256, 256), (65536, 256, 256), (1024, 128, 256)]


@pytest.fixture(scope="module")
def ctx():
    from diamond import _native as N
    return N.get_context(0)


def ref_forward(A, W, b):
    return torch.tanh(A.double() @ W.double().T + b.double())


@pytest.mark.parametrize("c", [1e-3, 1.0, 10.0])
@pytest.mark.parametrize("M,N,K", SHAPES)
def test_f16_pair_forward_vs_fp64(ctx, M, N, K, c):
    """A = tanh(randn * c): tiny, moderate and saturated activations; the shapes cover full, half-width tail and small-problem
    (every tile split) schedules and a clipped last row tile."""
    g = torch.Generator(device="cuda").manual_seed(M + N + K + int(c * 1000))
    A = torch.tanh(torch.randn(M, K, device="cuda", generator=g) * c)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    C = ctx.tc_linear_forward(F16, A, W, b)
    assert (C.double() - ref_forward(A, W, b)).abs().max().item() <= TC_TOL


def test_f16_pair_forward_per_row_weight_scales(ctx):
    """Row magnitudes from 2^-20 to 2^8 and all-zero rows: each row keeps its relative accuracy (without a per-row scale the small
    rows would fall into fp16's subnormal range).  With a zero bias, tanh(z) ~ z for the small rows, so their outputs carry the
    error of the products, which is bounded relative to the row's sum of |a w| (tanh' <= 1 for the large rows)."""
    M, N, K = 4096, 256, 256
    g = torch.Generator(device="cuda").manual_seed(5)
    A = torch.tanh(torch.randn(M, K, device="cuda", generator=g))
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    e = torch.linspace(-20, 8, N, device="cuda")
    W = W * torch.exp2(e)[:, None]
    W[::17] = 0.0
    b = torch.zeros(N, device="cuda")
    C = ctx.tc_linear_forward(F16, A, W, b).double()
    ref = ref_forward(A, W, b)
    S = A.double().abs() @ W.double().abs().T
    assert torch.all(C[:, ::17] == 0.0)
    assert torch.all((C - ref).abs() <= 1e-5 * S + 1e-6 * ref.abs())


def test_f16_pair_forward_non_finite_weights_match_the_tf32_path(ctx):
    """A NaN or Inf weight makes its row's pre-activations NaN in both formats (fp16: lo = Inf - Inf; TF32: the rounded hi of Inf
    is a NaN pattern); the epilogue then gives what the 3xTF32 path gives, bit for bit.  The other rows are unaffected."""
    M, N, K = 4096, 256, 256
    g = torch.Generator(device="cuda").manual_seed(6)
    A = torch.tanh(torch.randn(M, K, device="cuda", generator=g))
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    W[3, 7] = float("nan")
    W[100, 0] = float("inf")
    W[200, 255] = -float("inf")
    C = ctx.tc_linear_forward(F16, A, W, b)
    C32 = ctx.tc_linear_forward(0, A, W, b)
    bad = [3, 100, 200]
    assert torch.equal(C[:, bad].nan_to_num(nan=7.0), C32[:, bad].nan_to_num(nan=7.0))
    good = torch.ones(N, dtype=torch.bool, device="cuda")
    good[bad] = False
    assert torch.isfinite(C[:, good]).all()
    assert (C[:, good].double() - ref_forward(A, W[good], b[good])).abs().max().item() <= TC_TOL


@pytest.mark.parametrize("rows", [0, 1, 2500, 5000, 8192, 9000])
def test_f16_pair_forward_device_row_count(ctx, rows):
    """The row count read on the device (dppo_mlp_next_values): rows below it are computed, 256-row tiles past it are never
    written."""
    M, N, K = 8192, 256, 256
    g = torch.Generator(device="cuda").manual_seed(7)
    A = torch.tanh(torch.randn(M, K, device="cuda", generator=g))
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    out = torch.full((M, N), 7.0, device="cuda")
    m_dev = torch.tensor([rows], dtype=torch.int32, device="cuda")
    C = ctx.tc_linear_forward(F16, A, W, b, rows_dev=m_dev, out=out)
    r = min(rows, M)
    if r:
        assert (C[:r].double() - ref_forward(A[:r], W, b)).abs().max().item() <= TC_TOL
    assert torch.all(C[(r + 255) // 256 * 256:] == 7.0)


def test_f16_pair_forward_refuses_other_formats(ctx):
    from diamond import _native as N
    A = torch.zeros(1024, 256, device="cuda")
    W = torch.zeros(256, 256, device="cuda")
    b = torch.zeros(256, device="cuda")
    with pytest.raises(N.NativeError):
        ctx.tc_linear_forward(2, A, W, b)


@pytest.mark.parametrize("gemm_heads", [False, True])
@pytest.mark.parametrize("M", [4096, 5000, 19200])
def test_f16_pair_training_step_matches_fp32_path(ctx, M, gemm_heads):
    """One minibatch gradient at H = 256 (forward layers 2 and 3 on fp16 pairs) against the FFMA path, to the bound the 3xTF32
    path is held to (test_tensor_core_training_step_matches_fp32_path)."""
    from diamond import _native as N
    from diamond.flat import FlatMlp
    from test_kernels_gpu import dev, make_hyper, nerr, rand_params
    D, H, A = 64, 256, 4
    B = 2 * M
    rng = np.random.default_rng(M + 3)
    p = rand_params(rng, O.DISCRETE_PARAM_NAMES, D, H, A, False)
    fm = FlatMlp(D, H, A, False)
    flat = fm.pack(p, device="cuda")
    obs = dev(rng.standard_normal((B, D)).astype(np.float32)); act = dev(rng.integers(0, A, B), torch.int32)
    old_lp = dev((rng.standard_normal(B) * 0.3 - 1.0).astype(np.float32))
    adv = dev(rng.standard_normal(B).astype(np.float32)); ret = dev(rng.standard_normal(B).astype(np.float32))
    idx = dev(rng.permutation(B)[:M].astype(np.int32), torch.int32)
    hyper, _ = make_hyper(N, M)
    nb = ctx.mlp_gemm_heads_workspace_bytes(fm.desc, M) if gemm_heads else ctx.mlp_workspace_bytes(fm.desc, M, True)
    ws = torch.empty(nb // 4 + 512, device="cuda")
    fn = ctx.mlp_grad_minibatch_gemm_heads if gemm_heads else ctx.mlp_grad_minibatch
    out = {}
    try:
        for tc in (1, 0):
            ctx.set_option("tensor_cores", tc)
            grads = torch.zeros(fm.total, device="cuda"); losses = torch.zeros(4, device="cuda")
            fn(fm.desc, flat, grads, obs, act, old_lp, adv, ret, None, idx, M, hyper, losses, ws)
            torch.cuda.synchronize()
            out[tc] = (grads.cpu().numpy(), losses.cpu().numpy())
    finally:
        ctx.set_option("tensor_cores", 1)
    np.testing.assert_allclose(out[1][1], out[0][1], rtol=1e-5, atol=1e-7)
    gv, gv0 = fm.views(torch.as_tensor(out[1][0])), fm.views(torch.as_tensor(out[0][0]))
    for n in O.DISCRETE_PARAM_NAMES:
        assert nerr(gv[n].numpy(), gv0[n].numpy()) <= 2e-5, n
