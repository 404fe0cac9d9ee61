"""Projected sequence head (csrc/gru.cu: k_gru_xproj / k_gru_xwgrad; sldm_gnn_b200/gru.py: gru_projected_last_hidden):
layer 0 fed through an input projection x -> gi, so sequences longer, or inputs wider, than layer 0's shared-memory
x tile still run on the fused kernels.

Same bar as tests/test_gru.py and tests/test_gru_stack.py: fp32 rtol 1e-5 / atol 1e-6 against torch's CPU GRU
(parameter gradients with atol scaled by their magnitude), elements outside it adjudicated against the fp64 run.
Every GPU case aimed at the projected path asserts that the tile stack does not cover it, so that a carelessly chosen
shape cannot test the tile path instead.
"""
import copy

import pytest
import torch

import sldm_gnn_b200 as sg
from sldm_gnn_b200 import _lib
from sldm_gnn_b200.gru import (fused_gru_eligible, fused_gru_projected_eligible, fused_gru_stack_eligible,
                               gru_projected_last_hidden, gru_stack_last_hidden)
from test_gru_stack import _check_against_cpu

CAP = 128   # kGruMaxProjI: the widest layer-0 input of the projected path (W_ih is held in shared memory)


def _fwd_launches(L):
    return 2 * L


def _launches(L):
    """forward 2L, backward 3 + 4(L-1)"""
    return 2 * L + 3 + 4 * (L - 1)


def _projected_only(gru, x):
    return fused_gru_projected_eligible(gru, x) and not fused_gru_stack_eligible(gru, x)


# ------------------------------------------------------------------- CPU side --
def test_projected_support_query_without_gpu():
    lib = _lib.lib
    for I, H in ((6, 96), (9, 96), (64, 32), (CAP, 96), (1, 64)):
        assert lib.sldm_gru_projected_supported(I, H) == 1, (I, H)
    for I, H in ((6, 48), (6, 128), (0, 96), (CAP + 1, 96), (CAP + 1, 32)):
        assert lib.sldm_gru_projected_supported(I, H) == 0, (I, H)
    # the existing queries keep their limits
    assert lib.sldm_gru_supported(16, 9, 96) == 0 and lib.sldm_gru_stack_supported(400, 8, 96) == 0


def test_projected_entry_points_validate_arguments_without_gpu():
    lib = _lib.lib
    E, V, W, OK = _lib.EUNSUPPORTED, _lib.EINVAL, _lib.EWORKSPACE, _lib.OK
    fwd = lambda N, T, I, H, x=None, w=None, b=None, gi=None: lib.sldm_gru_input_project_forward(x, N, T, I, H, w, b, gi, None)
    wg = lambda N, T, I, H, dgi=None, x=None, p=None, tiles=1 << 20: lib.sldm_gru_input_wgrad(dgi, x, N, T, I, H, p, tiles, None)
    for H in (16, 48, 128):
        assert fwd(4, 16, 6, H) == E and wg(4, 16, 6, H) == E
    assert fwd(4, 16, CAP + 1, 96) == E and wg(4, 16, CAP + 1, 96) == E
    with pytest.raises(NotImplementedError, match="input width"):
        _lib.check(fwd(4, 16, CAP + 1, 96))
    for N, T, I in ((-1, 16, 6), (4, 0, 6), (4, 16, 0)):
        assert fwd(N, T, I, 96) == V and wg(N, T, I, 96) == V
    assert fwd(4, 16, 6, 96) == V and wg(4, 16, 6, 96) == V                     # NULL pointers
    assert fwd(4, 16, 6, 96, x=16, w=16, b=16) == V                             # NULL gi
    assert wg(4, 16, 6, 96, dgi=16, x=16) == V                                  # NULL partials
    assert wg(4000, 64, 6, 96, dgi=16, x=16, p=16, tiles=1) == W                # too few partial tiles
    assert wg(4, 16, 6, 96, dgi=8, x=16, p=16) == V                             # dgi not 16-byte aligned
    assert fwd(0, 16, 6, 96) == OK and wg(0, 16, 6, 96) == OK                   # nothing to do
    assert fwd(0, 500, CAP, 32) == OK and wg(0, 500, CAP, 32) == OK


def test_cpu_tensors_are_not_projected_eligible_and_raise():
    gru = torch.nn.GRU(12, 96, 2, batch_first=True)
    x = torch.randn(4, 40, 12)
    assert not fused_gru_projected_eligible(gru, x)
    with pytest.raises(RuntimeError, match="CUDA only"):
        gru_projected_last_hidden(gru, x)


# ------------------------------------------------------------------- GPU side --
@pytest.mark.gpu
@pytest.mark.parametrize("N,T,I,H,L,need_dx", [
    (1, 31, 6, 96, 1, True), (65, 31, 6, 96, 1, True), (300, 200, 6, 96, 1, False), (130, 128, 6, 32, 2, True),
    (63, 90, 6, 64, 2, False), (1000, 16, 9, 96, 1, True), (257, 16, 16, 64, 3, False), (77, 5, 40, 96, 2, True),
    (33, 1, CAP, 96, 1, True), (4099, 48, 6, 96, 2, False),
])
def test_projected_gru_matches_torch_gru(N, T, I, H, L, need_dx):
    dev = torch.device("cuda:0")
    torch.manual_seed(N * 131 + T * 7 + I + H + L)
    gru = torch.nn.GRU(I, H, L, batch_first=True).to(dev)
    x = torch.randn(N, T, I, device=dev, requires_grad=need_dx)
    up = torch.randn(N, H, device=dev)
    assert _projected_only(gru, x)
    before = _lib.lib.sldm_launch_count()
    h = gru_projected_last_hidden(gru, x)
    assert _lib.lib.sldm_launch_count() - before == _fwd_launches(L)
    h.backward(up)
    torch.cuda.synchronize()
    assert _lib.lib.sldm_launch_count() - before == _launches(L)
    _check_against_cpu(gru, x, up, h, need_dx)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 2])
def test_projected_path_at_a_tile_shape_matches_torch_gru(L):
    """Called directly where the tile path also applies (777 x 16 x 6, hidden 96): within the bar of the CPU GRU.  The
    two fused paths sum the input product in different places, so they are not bit-equal to each other."""
    dev = torch.device("cuda:0")
    torch.manual_seed(70 + L)
    gru = torch.nn.GRU(6, 96, L, batch_first=True).to(dev)
    x = torch.randn(777, 16, 6, device=dev, requires_grad=True)
    up = torch.randn(777, 96, device=dev)
    assert fused_gru_projected_eligible(gru, x) and fused_gru_stack_eligible(gru, x)
    h = gru_projected_last_hidden(gru, x)
    h.backward(up)
    _check_against_cpu(gru, x, up, h, True)


@pytest.mark.gpu
def test_projected_inference_equals_training_forward_and_is_deterministic():
    dev = torch.device("cuda:0")
    torch.manual_seed(5)
    gru = torch.nn.GRU(6, 96, 2, batch_first=True).to(dev)
    x = torch.randn(777, 40, 6, device=dev)
    up = torch.randn(777, 96, device=dev)
    assert _projected_only(gru, x)
    with torch.no_grad():
        h0 = gru_projected_last_hidden(gru, x)
    with torch.inference_mode():
        h1 = gru_projected_last_hidden(gru, x)
    grads = []
    for _ in range(2):
        gru.zero_grad()
        h2 = gru_projected_last_hidden(gru, x)
        h2.backward(up)
        grads.append([p.grad.clone() for p in gru.parameters()])
    assert torch.equal(h0, h1) and torch.equal(h0, h2.detach())
    assert all(torch.equal(a, b) for a, b in zip(*grads)), "parameter gradients are bit-identical run to run"


def _grusage(F, T, H, L, dev):
    torch.manual_seed(13 + F + T + L)
    return sg.GruSage(dynamic_features_num=F, frames_num=T, gru_hidden_size=H, gru_num_layers=L, fc1dims=[96],
                      sage_hidden_dims=[96, 96], fc2dims=[32], dropout=None, negative_slope=0.1,
                      map_included=False).to(dev)


@pytest.mark.gpu
@pytest.mark.parametrize("F,T,L", [(6, 48, 1), (12, 16, 2)])
def test_grusage_routes_a_long_or_wide_head_to_the_projected_path(monkeypatch, F, T, L):
    dev = torch.device("cuda:0")
    m = _grusage(F, T, 96, L, dev)
    x = torch.randn(500, T, F, device=dev)
    up = torch.randn(500, 96, device=dev)
    assert _projected_only(m.gru, x) and not fused_gru_eligible(m.gru, x)
    before = _lib.lib.sldm_launch_count()
    h = m._last_hidden(x)
    assert _lib.lib.sldm_launch_count() - before == _fwd_launches(L)
    h.backward(up)
    torch.cuda.synchronize()
    assert _lib.lib.sldm_launch_count() - before == _launches(L)
    ours = {k: p.grad.clone() for k, p in m.gru.named_parameters()}
    m.zero_grad(set_to_none=True)
    monkeypatch.setenv("SLDM_DISABLE_FUSED_GRU", "1")
    before = _lib.lib.sldm_launch_count()
    h_lib = m._last_hidden(x)
    h_lib.backward(up)
    torch.cuda.synchronize()
    assert _lib.lib.sldm_launch_count() == before
    assert torch.allclose(h, h_lib, rtol=1e-5, atol=2e-6), float((h - h_lib).abs().max())
    for k, p in m.gru.named_parameters():
        scale = max(1.0, float(p.grad.abs().max()))
        assert torch.allclose(ours[k], p.grad, rtol=1e-4, atol=2e-6 * scale), (k, float((ours[k] - p.grad).abs().max()))


def _small_model(dev, features, seed):
    """A small full model (map encoder + attention + a one-layer hidden-32 GRU head over `features` dynamic features,
    more than the x tile takes) and a batch builder, as in test_gru_stack."""
    from types import SimpleNamespace
    g = torch.Generator().manual_seed(400 + seed)
    S = 48
    mt = dict(float_features=torch.randn(S, 6, generator=g), bool_features=torch.rand(S, 3, generator=g) > 0.5,
              lane_type_cats=torch.randint(0, 4, (S,), generator=g),
              mgraph_edge_indexes=torch.stack([torch.randint(0, S, (4 * S,), generator=g), torch.randint(0, S, (4 * S,), generator=g)]),
              mseg_centroids=torch.rand(S, 2, generator=g) * 100.0)
    kw = dict(dynamic_features_num=features, frames_num=8, gru_hidden_size=32, gru_num_layers=1, fc1dims=[24],
              sage_hidden_dims=[32, 32], fc2dims=[16], out_dim=1, num_st_types=9, emb_dim=4, dropout=None,
              negative_slope=0.1, global_pooling="double", mapenc_lane_embdim=4, mapenc_sage_hdims=[16, 16],
              map_attention_topk=3)
    torch.manual_seed(seed)
    model = sg.GruSage(**kw, map_tensors=mt).to(dev)

    def batch(graphs, s):
        gg = torch.Generator().manual_seed(s)
        ns = [int(torch.randint(4, 11, (1,), generator=gg)) for _ in range(graphs)]
        off, eis, bv = 0, [], []
        for i, n in enumerate(ns):
            src = torch.randint(0, n, (3 * n,), generator=gg)
            eis.append(torch.stack([src, (src + 1 + torch.randint(0, n - 1, (3 * n,), generator=gg)) % n]) + off)
            bv += [i] * n
            off += n
        N = off
        d = dict(x=torch.randn(N, 8, features, generator=gg), xdims=torch.randn(N, 2, generator=gg),
                 xsttype=torch.randint(0, 9, (N,), generator=gg), pos_raw=torch.rand(N, 8, 2, generator=gg) * 100.0,
                 edge_index=torch.cat(eis, 1), batch=torch.tensor(bv), y=(torch.rand(graphs, 1, generator=gg) > 0.5).float())
        return SimpleNamespace(**{k: v.to(dev) for k, v in d.items()}, num_graphs=graphs)

    return model, batch


@pytest.mark.gpu
def test_graphed_grusage_with_a_projected_head_matches_the_uncaptured_model():
    from sldm_gnn_b200.grusage import GraphedGruSage
    dev = torch.device("cuda:0")
    model, batch = _small_model(dev, 10, seed=0)
    crit = torch.nn.BCEWithLogitsLoss()
    g = GraphedGruSage(model, max_nodes=128, max_edges=512, max_graphs=12, training=True)
    for graphs, seed in ((11, 1), (5, 2), (8, 3)):
        data = batch(graphs, seed)
        assert _projected_only(model.gru, data.x)
        model.zero_grad(set_to_none=True)
        ref_logits = model(data)
        crit(ref_logits, data.y).backward()
        ref = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
        model.zero_grad(set_to_none=True)
        out = g(data)
        assert torch.allclose(out, ref_logits, rtol=1e-5, atol=1e-6), float((out - ref_logits).abs().max())
        crit(out, data.y).backward()
        got = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}
        assert set(got) == set(ref) and "gru.weight_ih_l0" in got
        for k in ref:
            scale = max(1.0, float(ref[k].abs().max()))
            assert torch.allclose(got[k], ref[k], rtol=1e-4, atol=2e-6 * scale), (k, float((got[k] - ref[k]).abs().max()))


@pytest.mark.gpu
def test_graphed_train_step_with_a_projected_head_follows_the_eager_loop():
    import torch.nn.functional as Fn
    from sldm_gnn_b200.grusage import GraphedTrainStep
    dev = torch.device("cuda:0")
    model, batch = _small_model(dev, 10, seed=2)
    twin = copy.deepcopy(model)
    pw = torch.tensor(1.5, device=dev)
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=pw)
    loss_fn = lambda logits, y, w: Fn.binary_cross_entropy_with_logits(logits, y, weight=w, pos_weight=pw, reduction="sum")
    opt_e = torch.optim.Adam(twin.parameters(), lr=1e-3, weight_decay=5e-5)
    opt_g = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=5e-5, capturable=True)
    step = GraphedTrainStep(model, opt_g, loss_fn, max_nodes=128, max_edges=512, max_graphs=12)
    losses_e, losses_g = [], []
    for i, (graphs, seed) in enumerate(((11, 1), (5, 2), (8, 3), (11, 4), (3, 5), (9, 6))):
        data = batch(graphs, seed)
        assert _projected_only(model.gru, data.x)
        opt_e.zero_grad()
        le = crit(twin(data), data.y)
        le.backward()
        lg = step(data, data.y)
        if i == 0:
            ge = dict(twin.named_parameters())
            for k, p in model.named_parameters():
                scale = max(1.0, float(ge[k].grad.abs().max()))
                assert torch.allclose(p.grad, ge[k].grad, rtol=1e-4, atol=2e-6 * scale), (k, float((p.grad - ge[k].grad).abs().max()))
        opt_e.step()
        losses_e.append(float(le)); losses_g.append(float(lg))
    assert all(abs(a - b) <= 2e-3 * max(1.0, abs(a)) for a, b in zip(losses_e, losses_g)), (losses_e, losses_g)


@pytest.mark.gpu
def test_modules_outside_the_projected_range_stay_on_the_library():
    dev = torch.device("cuda:0")
    x = torch.randn(8, 40, 6, device=dev)
    assert not fused_gru_projected_eligible(torch.nn.GRU(6, 128, 1, batch_first=True).to(dev), x)
    assert not fused_gru_projected_eligible(torch.nn.GRU(6, 96, 1, batch_first=True, bidirectional=True).to(dev), x)
    assert not fused_gru_projected_eligible(torch.nn.GRU(6, 96, 1, batch_first=False).to(dev), x)
    assert not fused_gru_projected_eligible(torch.nn.GRU(6, 96, 1, batch_first=True).to(dev), x.double())
    drop = torch.nn.GRU(6, 96, 2, batch_first=True, dropout=0.2).to(dev)
    assert not fused_gru_projected_eligible(drop, x)                 # inter-layer dropout while training
    assert fused_gru_projected_eligible(drop.eval(), x)              # ... is inactive in eval()
    wide = torch.randn(8, 16, CAP + 1, device=dev)
    assert not fused_gru_projected_eligible(torch.nn.GRU(CAP + 1, 96, 1, batch_first=True).to(dev), wide)
    with pytest.raises(NotImplementedError):
        gru_projected_last_hidden(torch.nn.GRU(6, 128, 1, batch_first=True).to(dev), x)
    for F, H, L, xin, dropout in ((6, 128, 1, x, 0.0), (CAP + 1, 96, 1, wide, 0.0), (6, 96, 2, x, 0.2)):
        m = _grusage(F, xin.size(1), H, L, dev)
        m.gru.dropout = dropout
        before = _lib.lib.sldm_launch_count()
        m._last_hidden(xin)
        assert _lib.lib.sldm_launch_count() == before, (F, H, L, dropout)


@pytest.mark.gpu
def test_projected_gru_at_a_larger_shape():
    """About 20 k sequences of 64 frames x 6 features, hidden 96, two layers: full parity including dx."""
    dev = torch.device("cuda:0")
    torch.manual_seed(21)
    gru = torch.nn.GRU(6, 96, 2, batch_first=True).to(dev)
    x = torch.randn(20011, 64, 6, device=dev, requires_grad=True)
    up = torch.randn(20011, 96, device=dev)
    assert _projected_only(gru, x)
    h = gru_projected_last_hidden(gru, x)
    h.backward(up)
    _check_against_cpu(gru, x, up, h, True)


@pytest.mark.gpu
def test_projected_gru_inference_past_32_bit_offsets():
    """120 000 x 64 x 6 at hidden 96: gi has N*T*3H = 2.2e9 elements (8.8 GB), past 2^31.  Compared with torch's
    native GPU GRU (cuDNN off, run in slices as GruSage._last_hidden does) at the bar of the routing tests."""
    dev = torch.device("cuda:0")
    torch.manual_seed(22)
    N, T, I, H = 120000, 64, 6, 96
    assert N * T * 3 * H > 2 ** 31
    gru = torch.nn.GRU(I, H, 1, batch_first=True).to(dev)
    x = torch.randn(N, T, I, device=dev)
    assert _projected_only(gru, x)
    with torch.no_grad():
        before = _lib.lib.sldm_launch_count()
        h = gru_projected_last_hidden(gru, x)
        assert _lib.lib.sldm_launch_count() - before == 2
        rows = (1 << 30) // (T * 3 * H)
        with torch.backends.cudnn.flags(enabled=False):
            want = torch.cat([gru(x[i:i + rows])[1][-1] for i in range(0, N, rows)], dim=0)
    assert torch.allclose(h, want, rtol=1e-5, atol=2e-6), float((h - want).abs().max())
