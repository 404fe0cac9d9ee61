"""Stacked sequence head (nn.GRU(num_layers = L), GruSage(gru_num_layers > 1)) on the fused kernels of csrc/gru.cu
(sldm_gnn_b200/gru.py: gru_stack_last_hidden) against the reference's own layer, torch's CPU GRU.

Same bar as tests/test_gru.py: fp32 rtol 1e-5 / atol 1e-6 (parameter gradients with atol scaled by their magnitude),
elements outside it adjudicated against the fp64 run.  The numpy oracle of the stack lives here: layer by layer it is
the single-layer oracle of oracle/gru_oracle.py, plus the per-step upstream gradient a lower layer receives.
"""
import copy
import os

import numpy as np
import pytest
import torch

import sldm_gnn_b200 as sg
from sldm_gnn_b200 import _lib
from sldm_gnn_b200.gru import (fused_gru_eligible, fused_gru_stack_eligible, gru_last_hidden,
                               gru_stack_last_hidden)
from test_gru import _close

GOLDEN = sorted(__import__("glob").glob(os.path.join(os.path.dirname(__file__), "golden", "gru_stack", "*.pt")))


def _launches(L):
    """forward 1 + 2(L-1), backward 2 + 4(L-1)"""
    return 3 + 6 * (L - 1)


# ----------------------------------------------------------------- numpy oracle --
def stack_forward_oracle(x, layers):
    """layers: [(W_ih, W_hh, b_ih, b_hh)] per layer.  Returns (h_last of the top layer, tapes, output sequences)."""
    from oracle.gru_oracle import gru_last_hidden_oracle
    inp, tapes, seqs = np.asarray(x), [], []
    for W_ih, W_hh, b_ih, b_hh in layers:
        h, tape = gru_last_hidden_oracle(inp, W_ih, W_hh, b_ih, b_hh)
        T = inp.shape[1]
        seq = np.stack([tape[t + 1][0] for t in range(T - 1)] + [h], axis=1)      # h_t = h_prev of step t+1
        tapes.append(tape)
        seqs.append(seq)
        inp = seq
    return inp[:, -1, :], tapes, seqs


def stack_backward_oracle(dh_last, x, layers, tapes, seqs):
    """Returns (dx, [(dW_ih, dW_hh, db_ih, db_hh)] per layer).  The top layer starts from dh_last; layer l < L-1 starts
    from zeros and receives dY_l[t] = dgi_{l+1}[t] W_ih_{l+1} at the top of step t."""
    L = len(layers)
    dy, grads = None, [None] * L
    for l in range(L - 1, -1, -1):
        W_ih, W_hh = layers[l][0], layers[l][1]
        inp = np.asarray(x) if l == 0 else seqs[l - 1]
        N, T, _ = inp.shape
        H = W_hh.shape[1]
        dh = np.asarray(dh_last).copy() if l == L - 1 else np.zeros((N, H), dtype=inp.dtype)
        dinp = np.zeros_like(inp)
        dW_ih, dW_hh = np.zeros_like(W_ih), np.zeros_like(W_hh)
        db_ih, db_hh = np.zeros(3 * H, dtype=inp.dtype), np.zeros(3 * H, dtype=inp.dtype)
        for t in range(T - 1, -1, -1):
            if dy is not None:
                dh = dh + dy[:, t, :]
            h_prev, r, z, n, hn = tapes[l][t]
            dz = dh * (h_prev - n) * (1.0 - z) * z
            dn = dh * (1.0 - z) * (1.0 - n * n)
            dhn = dn * r
            dr = dn * hn * (1.0 - r) * r
            dgi = np.concatenate([dr, dz, dn], axis=1)
            dgh = np.concatenate([dr, dz, dhn], axis=1)
            dW_ih += dgi.T @ inp[:, t, :]
            dW_hh += dgh.T @ h_prev
            db_ih += dgi.sum(axis=0)
            db_hh += dgh.sum(axis=0)
            dinp[:, t, :] = dgi @ W_ih
            dh = dh * z + dgh @ W_hh
        grads[l] = (dW_ih, dW_hh, db_ih, db_hh)
        dy = dinp
    return dy, grads


def _torch_stack(c, state_dict, dt):
    g = torch.nn.GRU(c["I"], c["H"], c["L"], batch_first=True).to(dt)
    g.load_state_dict({k: v.to(dt) for k, v in state_dict.items()})
    return g


# ------------------------------------------------------------------- CPU side --
def test_stack_support_queries_without_gpu():
    lib = _lib.lib
    assert lib.sldm_gru_stack_supported(16, 6, 96) == 1 and lib.sldm_gru_stack_supported(1, 1, 32) == 1
    assert lib.sldm_gru_stack_supported(16, 8, 64) == 1 and lib.sldm_gru_stack_supported(100, 1, 96) == 1
    assert lib.sldm_gru_stack_supported(16, 6, 128) == 0     # hidden size outside the tile design
    assert lib.sldm_gru_stack_supported(16, 9, 96) == 0      # layer 0's input too wide
    assert lib.sldm_gru_stack_supported(400, 8, 96) == 0     # layer 0's x tile does not fit shared memory
    assert lib.sldm_gru_stack_supported(0, 6, 96) == 0


@pytest.mark.parametrize("H", [16, 48, 128])
def test_stack_entry_points_reject_other_hidden_sizes_without_gpu(H):
    lib = _lib.lib
    E = _lib.EUNSUPPORTED
    assert lib.sldm_gru_layer_forward(None, None, 4, 16, 6, H, None, None, None, None, None, None, None, None) == E
    assert lib.sldm_gru_layer_forward(None, 8, 4, 500, 6, H, None, None, None, None, None, None, None, None) == E
    assert lib.sldm_gru_layer_backward(None, 4, 16, 6, H, *([None] * 8), 1, None) == E
    assert lib.sldm_gru_project_forward(None, 64, H, None, None, None, None) == E
    assert lib.sldm_gru_project_backward(None, 64, H, None, None, None) == E
    assert lib.sldm_gru_wgrad_strided(None, None, H, 4, 16, H, None, 1, None) == E
    with pytest.raises(NotImplementedError, match=f"hidden size {H}"):
        _lib.check(lib.sldm_gru_project_forward(None, 64, H, None, None, None, None))


def test_stack_entry_points_validate_arguments_without_gpu():
    lib = _lib.lib
    assert lib.sldm_gru_layer_forward(None, None, -1, 16, 6, 96, None, None, None, None, None, None, None, None) == _lib.EINVAL
    assert lib.sldm_gru_project_forward(None, -1, 96, None, None, None, None) == _lib.EINVAL
    assert lib.sldm_gru_wgrad_strided(None, None, 98, 4, 16, 96, None, 1, None) == _lib.EINVAL   # stride not a multiple of 4
    assert lib.sldm_gru_wgrad_strided(None, None, 32, 4, 16, 96, None, 1, None) == _lib.EINVAL   # stride < H
    # deep mode (gi given): no shared-memory limit on T, so T = 500 is not refused -- only the NULL pointers are
    assert lib.sldm_gru_layer_forward(None, 16, 4, 500, 6, 96, None, None, None, None, None, None, None, None) == _lib.EINVAL
    for fn, args in ((lib.sldm_gru_layer_forward, (None, None, 0, 16, 6, 96) + (None,) * 8),
                     (lib.sldm_gru_project_backward, (None, 0, 96, None, None, None))):
        assert fn(*args) == _lib.OK                                                          # nothing to do


def test_cpu_tensors_are_not_stack_eligible_and_raise():
    gru = torch.nn.GRU(6, 96, 2, batch_first=True)
    x = torch.randn(4, 16, 6)
    assert not fused_gru_stack_eligible(gru, x)
    with pytest.raises(RuntimeError, match="CUDA only"):
        gru_stack_last_hidden(gru, x)


def test_stack_golden_files_exist():
    assert len(GOLDEN) == 3


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-3] for p in GOLDEN])
def test_stack_golden_fixtures_are_what_torch_gru_computes(path):
    fix = torch.load(path)
    c = fix["cfg"]
    g = _torch_stack(c, fix["state_dict"], torch.float32)
    x = fix["x"].clone().requires_grad_(True)
    h = g(x)[1][-1]
    h.backward(fix["up"])
    assert torch.allclose(h, fix["f32"]["h"], rtol=1e-6, atol=1e-7)
    assert torch.allclose(x.grad, fix["f32"]["dx"], rtol=1e-5, atol=1e-6)
    for k, p in g.named_parameters():
        want = fix["f32"]["grads"][k]
        assert torch.allclose(p.grad, want, rtol=1e-5, atol=1e-6 * max(1.0, float(want.abs().max()))), k


def _oracle_run(x, sd, L, up):
    layers = [tuple(sd[f"{k}_l{l}"] for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")) for l in range(L)]
    h, tapes, seqs = stack_forward_oracle(x, layers)
    dx, grads = stack_backward_oracle(up, x, layers, tapes, seqs)
    got = {}
    for l, gl in enumerate(grads):
        got.update({f"{k}_l{l}": v for k, v in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), gl)})
    return h, dx, got


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-3] for p in GOLDEN])
def test_numpy_stack_oracle_reproduces_the_golden_vectors(path):
    fix = torch.load(path)
    sd = {k: v.double().numpy() for k, v in fix["state_dict"].items()}
    h, dx, got = _oracle_run(fix["x"].double().numpy(), sd, fix["cfg"]["L"], fix["up"].double().numpy())
    want = fix["f64"]
    assert abs(h - want["h"].numpy()).max() < 1e-12
    for k, g in got.items():
        w = want["grads"][k].numpy()
        assert abs(g - w).max() <= 1e-10 * max(1.0, abs(w).max()), k
    assert abs(dx - want["dx"].numpy()).max() < 1e-10


@pytest.mark.parametrize("L", [2, 3])
def test_numpy_stack_oracle_matches_torch_gru_in_fp64(L):
    torch.manual_seed(50 + L)
    c = dict(I=5, H=32, L=L)
    g = torch.nn.GRU(5, 32, L, batch_first=True).double()
    x = torch.randn(7, 6, 5, dtype=torch.float64, requires_grad=True)
    up = torch.randn(7, 32, dtype=torch.float64)
    h_t = g(x)[1][-1]
    h_t.backward(up)
    sd = {k: v.detach().numpy() for k, v in g.state_dict().items()}
    h, dx, got = _oracle_run(x.detach().numpy(), sd, c["L"], up.numpy())
    assert abs(h - h_t.detach().numpy()).max() < 1e-12
    for k, p in g.named_parameters():
        w = p.grad.numpy()
        assert abs(got[k] - w).max() <= 1e-10 * max(1.0, abs(w).max()), k
    assert abs(dx - x.grad.numpy()).max() < 1e-10


# ------------------------------------------------------------------- GPU side --
def _reference(gru, x, up, need_dx):
    """torch's own GRU stack on the CPU, fp32 and fp64: (h, grads, dx) each."""
    out = []
    for dt in (torch.float32, torch.float64):
        g = torch.nn.GRU(gru.input_size, gru.hidden_size, gru.num_layers, batch_first=True).to(dt)
        g.load_state_dict({k: v.detach().cpu().to(dt) for k, v in gru.state_dict().items()})
        xi = x.detach().cpu().to(dt).requires_grad_(need_dx)
        h = g(xi)[1][-1]
        h.backward(up.detach().cpu().to(dt))
        out.append((h.detach(), {k: p.grad for k, p in g.named_parameters()}, xi.grad))
    return out


def _check_against_cpu(gru, x, up, h, need_dx):
    (h32, g32, dx32), (h64, g64, dx64) = _reference(gru, x, up, need_dx)
    _close(h, h32, h64, "h_last")
    for k, p in gru.named_parameters():
        _close(p.grad, g32[k], g64[k], f"grad {k}", scale_atol=True)
    if need_dx:
        _close(x.grad, dx32, dx64, "dx")
    else:
        assert x.grad is None


@pytest.mark.gpu
@pytest.mark.parametrize("N,T,I,H,L,need_dx", [
    (1, 1, 1, 32, 2, False), (5, 3, 6, 96, 2, True), (65, 16, 6, 96, 2, True), (300, 7, 8, 64, 2, True),
    (130, 16, 3, 32, 4, False), (63, 25, 5, 96, 2, True), (1000, 16, 6, 96, 3, False), (4099, 16, 6, 96, 2, False),
])
def test_fused_gru_stack_matches_torch_gru(N, T, I, H, L, need_dx):
    dev = torch.device("cuda:0")
    torch.manual_seed(N * 131 + T * 7 + I + H + L)
    gru = torch.nn.GRU(I, H, L, batch_first=True).to(dev)
    x = torch.randn(N, T, I, device=dev, requires_grad=need_dx)
    up = torch.randn(N, H, device=dev)
    assert fused_gru_stack_eligible(gru, x) and not fused_gru_eligible(gru, x)
    before = _lib.lib.sldm_launch_count()
    h = gru_stack_last_hidden(gru, x)
    assert _lib.lib.sldm_launch_count() - before == 1 + 2 * (L - 1)
    h.backward(up)
    torch.cuda.synchronize()
    assert _lib.lib.sldm_launch_count() - before == _launches(L)
    _check_against_cpu(gru, x, up, h, need_dx)


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-3] for p in GOLDEN])
def test_fused_gru_stack_matches_golden(path):
    dev = torch.device("cuda:0")
    fix = torch.load(path)
    c = fix["cfg"]
    gru = _torch_stack(c, fix["state_dict"], torch.float32).to(dev)
    x = fix["x"].to(dev).requires_grad_(True)
    h = gru_stack_last_hidden(gru, x)
    h.backward(fix["up"].to(dev))
    _close(h, fix["f32"]["h"], fix["f64"]["h"], "h_last")
    _close(x.grad, fix["f32"]["dx"], fix["f64"]["dx"], "dx")
    for k, p in gru.named_parameters():
        _close(p.grad, fix["f32"]["grads"][k], fix["f64"]["grads"][k], f"grad {k}", scale_atol=True)


@pytest.mark.gpu
def test_fused_gru_stack_long_sequences():
    """T = 100: layer 0 (I = 1) still fits its x tile; the layers above have no shared-memory limit on T."""
    dev = torch.device("cuda:0")
    torch.manual_seed(100)
    gru = torch.nn.GRU(1, 96, 3, batch_first=True).to(dev)
    x = torch.randn(150, 100, 1, device=dev, requires_grad=True)
    up = torch.randn(150, 96, device=dev)
    assert fused_gru_stack_eligible(gru, x)
    h = gru_stack_last_hidden(gru, x)
    h.backward(up)
    _check_against_cpu(gru, x, up, h, True)


@pytest.mark.gpu
def test_fused_gru_stack_inference_equals_training_forward_and_is_deterministic():
    dev = torch.device("cuda:0")
    torch.manual_seed(4)
    gru = torch.nn.GRU(6, 96, 2, batch_first=True).to(dev)
    x = torch.randn(777, 16, 6, device=dev)
    up = torch.randn(777, 96, device=dev)
    with torch.no_grad():
        h0 = gru_stack_last_hidden(gru, x)
    with torch.inference_mode():
        h1 = gru_stack_last_hidden(gru, x)
    grads = []
    for _ in range(2):
        gru.zero_grad()
        h2 = gru_stack_last_hidden(gru, x)
        h2.backward(up)
        grads.append([p.grad.clone() for p in gru.parameters()])
    assert torch.equal(h0, h1) and torch.equal(h0, h2.detach())
    assert all(torch.equal(a, b) for a, b in zip(*grads)), "parameter gradients are bit-identical run to run"


@pytest.mark.gpu
def test_grusage_routes_a_stacked_head_to_the_kernels_and_matches_the_library(monkeypatch):
    dev = torch.device("cuda:0")
    torch.manual_seed(12)
    m = sg.GruSage(dynamic_features_num=6, frames_num=16, gru_hidden_size=96, gru_num_layers=2, fc1dims=[96],
                   sage_hidden_dims=[96, 96], fc2dims=[32], dropout=None, negative_slope=0.1,
                   map_included=False).to(dev)
    x = torch.randn(500, 16, 6, device=dev)
    up = torch.randn(500, 96, device=dev)
    before = _lib.lib.sldm_launch_count()
    h = m._last_hidden(x)
    assert _lib.lib.sldm_launch_count() - before == 3, "layer 0, then projection + recurrence of layer 1"
    h.backward(up)
    torch.cuda.synchronize()
    assert _lib.lib.sldm_launch_count() - before == _launches(2)
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


def _small_model(dev, layers, seed):
    """A small full model (map encoder + attention + a stacked GRU head) and a batch builder, as in test_grusage."""
    from types import SimpleNamespace
    g = torch.Generator().manual_seed(300 + seed)
    S = 48
    mt = dict(float_features=torch.randn(S, 6, generator=g), bool_features=torch.rand(S, 3, generator=g) > 0.5,
              lane_type_cats=torch.randint(0, 4, (S,), generator=g),
              mgraph_edge_indexes=torch.stack([torch.randint(0, S, (4 * S,), generator=g), torch.randint(0, S, (4 * S,), generator=g)]),
              mseg_centroids=torch.rand(S, 2, generator=g) * 100.0)
    kw = dict(dynamic_features_num=6, frames_num=8, gru_hidden_size=32, gru_num_layers=layers, fc1dims=[24],
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
        d = dict(x=torch.randn(N, 8, 6, generator=gg), xdims=torch.randn(N, 2, generator=gg),
                 xsttype=torch.randint(0, 9, (N,), generator=gg), pos_raw=torch.rand(N, 8, 2, generator=gg) * 100.0,
                 edge_index=torch.cat(eis, 1), batch=torch.tensor(bv), y=(torch.rand(graphs, 1, generator=gg) > 0.5).float())
        return SimpleNamespace(**{k: v.to(dev) for k, v in d.items()}, num_graphs=graphs)

    return model, batch


@pytest.mark.gpu
def test_graphed_grusage_with_a_stacked_head_matches_the_uncaptured_model():
    from sldm_gnn_b200.grusage import GraphedGruSage
    dev = torch.device("cuda:0")
    model, batch = _small_model(dev, 2, seed=0)
    crit = torch.nn.BCEWithLogitsLoss()
    g = GraphedGruSage(model, max_nodes=128, max_edges=512, max_graphs=12, training=True)
    for graphs, seed in ((11, 1), (5, 2), (8, 3)):
        data = batch(graphs, seed)
        assert fused_gru_stack_eligible(model.gru, data.x)
        model.zero_grad(set_to_none=True)
        ref_logits = model(data)
        crit(ref_logits, data.y).backward()
        ref = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
        model.zero_grad(set_to_none=True)
        out = g(data)
        assert torch.allclose(out, ref_logits, rtol=1e-5, atol=1e-6), float((out - ref_logits).abs().max())
        crit(out, data.y).backward()
        got = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}
        assert set(got) == set(ref) and any(k.startswith("gru.") and k.endswith("_l1") for k in got)
        for k in ref:
            scale = max(1.0, float(ref[k].abs().max()))
            assert torch.allclose(got[k], ref[k], rtol=1e-4, atol=2e-6 * scale), (k, float((got[k] - ref[k]).abs().max()))


@pytest.mark.gpu
def test_graphed_train_step_with_a_stacked_head_follows_the_eager_loop():
    import torch.nn.functional as Fn
    from sldm_gnn_b200.grusage import GraphedTrainStep
    dev = torch.device("cuda:0")
    model, batch = _small_model(dev, 2, seed=2)
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
def test_ineligible_stacks_stay_on_the_library():
    dev = torch.device("cuda:0")
    x = torch.randn(8, 16, 6, device=dev)
    drop = torch.nn.GRU(6, 96, 2, batch_first=True, dropout=0.2).to(dev)
    assert not fused_gru_stack_eligible(drop, x)                    # inter-layer dropout while training
    assert fused_gru_stack_eligible(drop.eval(), x)                 # ... is inactive in eval()
    assert not fused_gru_stack_eligible(torch.nn.GRU(6, 128, 2, batch_first=True).to(dev), x)
    assert not fused_gru_stack_eligible(torch.nn.GRU(6, 96, 2, batch_first=True, bidirectional=True).to(dev), x)
    assert not fused_gru_stack_eligible(torch.nn.GRU(6, 96, 2, batch_first=False).to(dev), x)
    assert not fused_gru_stack_eligible(torch.nn.GRU(6, 96, 2, batch_first=True).to(dev), x.double())
    with pytest.raises(NotImplementedError):
        gru_stack_last_hidden(torch.nn.GRU(6, 128, 2, batch_first=True).to(dev), x)
    m = sg.GruSage(dynamic_features_num=6, frames_num=16, gru_hidden_size=96, gru_num_layers=2, fc1dims=[96],
                   sage_hidden_dims=[96, 96], fc2dims=[32], dropout=None, negative_slope=0.1,
                   map_included=False).to(dev)
    m.gru.dropout = 0.2
    before = _lib.lib.sldm_launch_count()
    m._last_hidden(x)
    assert _lib.lib.sldm_launch_count() == before, "a training-mode stack with dropout runs on the library"


@pytest.mark.gpu
def test_fused_gru_stack_at_a_larger_shape():
    """About 20 k sequences of the reference's shape (16 frames x 6 features, hidden 96), two layers."""
    dev = torch.device("cuda:0")
    torch.manual_seed(20)
    gru = torch.nn.GRU(6, 96, 2, batch_first=True).to(dev)
    x = torch.randn(20011, 16, 6, device=dev, requires_grad=True)
    up = torch.randn(20011, 96, device=dev)
    h = gru_stack_last_hidden(gru, x)
    h.backward(up)
    _check_against_cpu(gru, x, up, h, True)
