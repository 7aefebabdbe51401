"""LSTM networks on the CPU: LSTMCore against torch.nn.LSTM, the cell = 1 parameter layout, the constructors' width rule, and a
mirror of the LSTM scan-branch choice in csrc/rnn.cu with the case table of tests/test_lstm_gpu.py.

The mirror restates rnn.cu's lstm_scan_blocks / lstm_cluster_plan so that the GPU case table can name, and this file can check, the
kernel each case runs: warp kernels at Hg = 8 / 16 / 32, tiled kernels with E environments per thread for the other multiples of 4
up to 96, cluster kernels with C CTAs and E environments per thread from 100 to 256."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from test_rnn_kernels_gpu import tiled_scan_E, tiled_scan_groups

# ---------------------------------------------------------------- mirror of the LSTM branch choice in csrc/rnn.cu --------------
SMEM_FLOATS = 227 * 1024 // 4                           # rnn.cu kScanSmemFloats
MAX_GROUPS = 8                                          # rnn.cu kClusterMaxGroups


def lstm_width_ok(Hg):                                  # rnn.cu lstm_width_ok
    return Hg % 4 == 0 and 8 <= Hg <= 256


def lstm_cluster_plan(N, Hg):
    """rnn.cu lstm_cluster_plan: (C, U, E, G, clusters)."""
    assert lstm_width_ok(Hg) and Hg > 96
    C = 4 if Hg <= 128 else 8
    U = -(-Hg // C)
    HP = (Hg + 3) & ~3
    fwd = lambda e: 4 * U * (HP + 4) + 2 * e * HP       # rnn.cu lstm_cluster_fwd_smem_floats
    bwd = lambda e: 4 * U * Hg + e * (4 * U + 2 * C * U)  # rnn.cu lstm_cluster_bwd_smem_floats
    cap = 1
    while fwd(cap + 1) <= SMEM_FLOATS and bwd(cap + 1) <= SMEM_FLOATS:
        cap += 1
    slots = 148 // C
    ec = min(-(-N // slots), cap, 4 * MAX_GROUPS)
    E = 1 if ec <= MAX_GROUPS else 2 if ec <= 2 * MAX_GROUPS else 4
    G = -(-ec // E)
    while G > 1 and G * E > cap:
        G -= 1
    return C, U, E, G, -(-N // (G * E))


def lstm_branch(N, Hg):
    """The forward / backward LSTM scan pair rnn.cu launches for (N, Hg)."""
    assert lstm_width_ok(Hg)
    if Hg in (8, 16, 32):
        return f"warp{Hg}"
    if Hg <= 96:
        return f"tiled{tiled_scan_E(N, Hg)}"
    C, U, E, G, _ = lstm_cluster_plan(N, Hg)
    return f"c{C}e{E}"


def lstm_envs_per_part(N, Hg):
    """Environments one scan block (warp / tiled) or cluster owns."""
    if Hg in (8, 16, 32):
        return 128 // Hg
    if Hg <= 96:
        E = tiled_scan_E(N, Hg)
        return tiled_scan_groups(N, Hg, E) * E
    C, U, E, G, _ = lstm_cluster_plan(N, Hg)
    return G * E


ALL_BRANCHES = {"warp8", "warp16", "warp32", "tiled1", "tiled2", "tiled4", "c4e1", "c4e2", "c4e4", "c8e1", "c8e2", "c8e4"}


def head_kernel(H, A):                                  # heads.cu launch_head_train_kernel (test_rnn_gaussian_gpu.head_kernel)
    return "split" if H in (128, 256) and A <= 4 else "generic"


# One row per case of tests/test_lstm_gpu.py: the branch, then the shapes.  N puts one environment in the last scan block or
# cluster wherever the branch allows it.  opts: "gauss" Gaussian policy (else categorical), "hx0" non-zero h0 and c0, "dones"
# resets (else prev_dones NULL), "norm" advantage normalisation from fp64 statistics, "den2" loss denominator 2 M.
CASES = [
    # id          branch    D    H   Hg  A   T     N   opts
    ("w8",        "warp8",  5, 128,   8, 3, 64,   17, "hx0 dones"),
    ("w8-g",      "warp8",  4,  32,   8, 2,  1,   17, "gauss hx0 dones"),
    ("w16",       "warp16", 4,  64,  16, 4, 33,    9, "hx0 dones norm"),
    ("w16-null",  "warp16", 4,  32,  16, 5, 33,   40, ""),
    ("w32",       "warp32", 8,  32,  32, 5, 33,    5, "hx0 dones den2"),
    ("w32-g",     "warp32", 6, 128,  32, 3,  2,    5, "gauss hx0 dones norm"),
    ("t12",       "tiled1", 6,  64,  12, 4, 33,   22, "hx0 dones"),
    ("t44-g",     "tiled1", 3, 200,  44, 2, 33,    7, "gauss hx0 dones den2"),
    ("t64",       "tiled1", 8,  64,  64, 4, 64,    5, "hx0 dones"),
    ("t64-e2",    "tiled2", 8,  64,  64, 4,  3, 1801, "hx0 dones norm"),
    ("t96",       "tiled1", 4, 128,  96, 3,  2,    3, "gauss hx0 dones"),
    ("t96-e4",    "tiled4", 4,  64,  96, 6,  2, 2369, "hx0 dones"),
    ("c100",      "c4e1",   4, 128, 100, 3, 33,   20, "hx0 dones"),
    ("c100-e2-g", "c4e2",   3,  64, 100, 2,  2,  331, "gauss hx0 dones norm"),
    ("c128-e4",   "c4e4",   5, 128, 128, 4,  3,  621, "hx0 dones den2"),
    ("c200-g",    "c8e1",   6, 128, 200, 2, 64,    5, "gauss hx0 dones"),
    ("c256-e2",   "c8e2",   3,  32, 256, 4,  2,  161, "hx0 dones norm"),
    ("c256-e4-g", "c8e4",   4,  64, 256, 3,  2,  321, "gauss dones"),
    ("c256",      "c8e1",   4,  64, 256, 5,  1,   19, "hx0 dones"),
]
CASE_IDS = [c[0] for c in CASES]


def test_lstm_case_table_covers_every_scan_instantiation():
    """Each case runs the branch it names; together they run every LSTM scan instantiation (warp 8 / 16 / 32, tiled E = 1 / 2 / 4,
    cluster C = 4 / 8 x E = 1 / 2 / 4), both policy kinds with both head kernels, T = 1, 2, odd and 64, and every option."""
    for cid, br, D, H, Hg, A, T, N, opts in CASES:
        assert lstm_branch(N, Hg) == br, cid
        if Hg > 96:
            C, U, E, G, _ = lstm_cluster_plan(N, Hg)
            assert U <= 32 and G * U <= 256, cid
    assert {c[1] for c in CASES} == ALL_BRANCHES
    one_past = {br for _, br, D, H, Hg, A, T, N, _ in CASES
                if N % lstm_envs_per_part(N, Hg) == 1 or lstm_envs_per_part(N, Hg) == 1}
    assert one_past == ALL_BRANCHES
    assert {1, 2, 64} <= {c[6] for c in CASES} and any(c[6] % 2 == 1 and c[6] > 16 for c in CASES)
    kinds = {("gauss" in c[8], head_kernel(c[3], c[5])) for c in CASES}
    assert kinds == {(False, "split"), (False, "generic"), (True, "split"), (True, "generic")}
    assert {"hx0", "dones", "norm", "den2", "gauss"} <= set(" ".join(c[8] for c in CASES).split())


def test_lstm_branch_rule():
    """The width rule and where the families meet: tiled up to 96, clusters of 4 CTAs up to 128 and of 8 up to 256."""
    assert [h for h in range(1, 300) if lstm_width_ok(h)] == list(range(8, 257, 4))
    assert lstm_branch(64, 96).startswith("tiled") and lstm_branch(64, 100) == "c4e1" and lstm_branch(64, 128) == "c4e1"
    assert lstm_branch(64, 132) == "c8e1" and lstm_branch(64, 256) == "c8e1"
    assert lstm_branch(4096, 64) == "tiled4" and lstm_branch(64, 64) == "tiled1"
    assert lstm_cluster_plan(4096, 256)[2] == 4 and lstm_cluster_plan(4096, 128)[2] == 4


# ---------------------------------------------------------------- LSTMCore against torch.nn.LSTM -------------------------------
@torch.no_grad()
def test_lstm_core_matches_torch_lstm_without_resets():
    from diamond.recurrent import LSTMCore
    torch.manual_seed(0)
    T, B, H, Hg = 7, 5, 6, 12
    core = LSTMCore(H, Hg).double()
    ref = torch.nn.LSTM(H, Hg).double()
    ref.load_state_dict(core.state_dict())
    x = torch.randn(T, B, H, dtype=torch.float64)
    h0, c0 = torch.randn(1, B, Hg, dtype=torch.float64), torch.randn(1, B, Hg, dtype=torch.float64)
    out, hx = core(x, torch.cat([h0, c0], -1), None)
    rout, (rh, rc) = ref(x, (h0, c0))
    assert hx.shape == (1, B, 2 * Hg)
    assert float((out - rout).abs().max()) <= 1e-6
    assert float((hx[..., :Hg] - rh).abs().max()) <= 1e-6 and float((hx[..., Hg:] - rc).abs().max()) <= 1e-6
    out0, hx0 = core(x, None, None)                     # hx None: zero state
    rout0, (rh0, rc0) = ref(x)
    assert float((out0 - rout0).abs().max()) <= 1e-6 and float((hx0 - torch.cat([rh0, rc0], -1)).abs().max()) <= 1e-6


@torch.no_grad()
def test_lstm_core_matches_stepwise_torch_lstm_with_resets():
    """Where dones[t] is set both h and c are zeroed before step t."""
    from diamond.recurrent import LSTMCore
    torch.manual_seed(1)
    T, B, H, Hg = 9, 6, 5, 8
    core = LSTMCore(H, Hg).double()
    ref = torch.nn.LSTM(H, Hg).double()
    ref.load_state_dict(core.state_dict())
    x = torch.randn(T, B, H, dtype=torch.float64)
    dones = torch.rand(T, B) < 0.3
    dones[0, 0] = True
    h, c = torch.randn(1, B, Hg, dtype=torch.float64), torch.randn(1, B, Hg, dtype=torch.float64)
    out, hx = core(x, torch.cat([h, c], -1), dones)
    outs = []
    for t in range(T):
        keep = (~dones[t]).double().view(1, B, 1)
        o, (h, c) = ref(x[t:t + 1], (h * keep, c * keep))
        outs.append(o[0])
    assert float((out - torch.stack(outs)).abs().max()) <= 1e-6
    assert float((hx - torch.cat([h, c], -1)).abs().max()) <= 1e-6


# ---------------------------------------------------------------- layout, slices and the constructors ---------------------------
@pytest.mark.parametrize("continuous", [0, 1])
def test_lstm_layout_and_slices(continuous):
    """cell = 1: the lstm.* tensors are 4 Hg rows, slices do not overlap, offsets are multiples of 4, the slice names and shapes are
    the LSTM network's, and the parameter count is the module's."""
    from diamond import _native as Nt
    from diamond.config import RecurrentContinuousPPOConfig, RecurrentPPOConfig
    from diamond.recurrent import RecurrentContinuousLSTMActorCriticNetwork, RecurrentLSTMActorCriticNetwork, rnn_param_slices
    D, H, Hg, A = 5, 64, 24, 3
    desc = Nt.RnnDesc(D, H, Hg, A, continuous, 1)
    lay = Nt.rnn_layout(desc)
    sl = rnn_param_slices(desc, lay)
    if continuous:
        net = RecurrentContinuousLSTMActorCriticNetwork(SimpleNamespace(shape=(D,)), SimpleNamespace(shape=(A,)),
                                                       RecurrentContinuousPPOConfig(network_hidden_dim=H, gru_hidden_dim=Hg))
    else:
        net = RecurrentLSTMActorCriticNetwork(SimpleNamespace(shape=(D,)), SimpleNamespace(n=A),
                                              RecurrentPPOConfig(network_hidden_dim=H, gru_hidden_dim=Hg))
    params = dict(net.named_parameters())
    assert {n: tuple(p.shape) for n, p in params.items()} == {n: shp for n, (off, shp) in sl.items()}
    assert sl["lstm.weight_hh_l0"][1] == (4 * Hg, Hg) and sl["lstm.bias_ih_l0"][1] == (4 * Hg,)
    spans = sorted((off, off + int(np.prod(shp))) for off, shp in sl.values())
    assert all(off % 4 == 0 for off, _ in spans)
    assert all(a_end <= b_off for (_, a_end), (b_off, _) in zip(spans, spans[1:]))
    assert spans[-1][1] <= lay.total < spans[-1][1] + 4
    assert sum(p.numel() for p in params.values()) == sum(int(np.prod(shp)) for _, shp in sl.values())
    # the GRU layout of the same descriptor is unchanged by the new field
    gru = Nt.rnn_layout(Nt.RnnDesc(D, H, Hg, A, continuous))
    assert gru.whh - gru.wih == (3 * Hg * H + 3) // 4 * 4 and "gru.weight_hh_l0" in rnn_param_slices(Nt.RnnDesc(D, H, Hg, A, continuous), gru)


@pytest.mark.parametrize("Hg", [4, 6, 10, 258, 260, 512])
def test_lstm_networks_refuse_unsupported_widths(Hg):
    from diamond.config import RecurrentContinuousPPOConfig, RecurrentPPOConfig
    from diamond.recurrent import RecurrentContinuousLSTMActorCriticNetwork, RecurrentLSTMActorCriticNetwork
    with pytest.raises(ValueError, match="multiple of 4 from 8 to 256"):
        RecurrentLSTMActorCriticNetwork(SimpleNamespace(shape=(4,)), SimpleNamespace(n=2), RecurrentPPOConfig(gru_hidden_dim=Hg))
    with pytest.raises(ValueError, match="multiple of 4 from 8 to 256"):
        RecurrentContinuousLSTMActorCriticNetwork(SimpleNamespace(shape=(3,)), SimpleNamespace(shape=(1,)),
                                                  RecurrentContinuousPPOConfig(gru_hidden_dim=Hg))


def test_lstm_networks_state_width_and_state_dict_keys():
    from diamond.config import RecurrentPPOConfig
    from diamond.recurrent import RecurrentLSTMActorCriticNetwork
    net = RecurrentLSTMActorCriticNetwork(SimpleNamespace(shape=(4,)), SimpleNamespace(n=2), RecurrentPPOConfig(gru_hidden_dim=16))
    assert net.recurrent_state_dim == 32
    assert {"lstm.weight_ih_l0", "lstm.weight_hh_l0", "lstm.bias_ih_l0", "lstm.bias_hh_l0"} <= set(net.state_dict())
    logits, values, hx = net.get_logits_values_and_hx(torch.randn(3, 2, 4), None, None)
    assert logits.shape == (3, 2, 2) and values.shape == (3, 2) and hx.shape == (1, 2, 32)
