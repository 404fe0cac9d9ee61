"""MapSpatialAttention with 9..32 nearest segments (GruSage `map_attention_topk` 9-32): the warp-per-vehicle kernels of
csrc/map_attention.cu (k_map_attention_grid_fwd_wide, k_map_attention_fwd_wide, k_map_attention_bwd_ds_wide,
k_map_attention_bwd_mlp_wide and k_map_attention_demb<9..32>).

Parity is against the oracle pinned to the reference class, adjudicated in fp64 as in tests/test_map_attention.py; the
grid search and the exhaustive scan must agree bit for bit; K <= 8 must still launch exactly the kernels it launched
before.  Run once as is (grid search) and once under SLDM_MAP_ATTENTION_SCAN=1 (exhaustive scan)."""
import copy
import re

import pytest
import torch

from oracle.grusage_oracle import GruSageOracle
from oracle.map_attention_oracle import MapSpatialAttentionOracle
from sldm_gnn_b200 import _lib
from test_grusage import GOLDEN as GRUSAGE_GOLDEN, Bag, _build, _step
from test_map_attention import _forward_raw, _geometries, _mask_clear

RTOL, ATOL = 1e-5, 1e-6


# ------------------------------------------------------------------------------ CPU --
def test_max_k_is_32():
    assert _lib.lib.sldm_map_attention_max_k() == 32


def test_workspace_query_by_k():
    q, qk = _lib.lib.sldm_map_attention_workspace_bytes, _lib.lib.sldm_map_attention_workspace_bytes_k
    for B in (0, 1, 1000, 205587):
        for H in (1, 16, 64):
            for K in range(1, 9):
                assert qk(B, H, K) == q(B, H), (B, H, K)
            sizes = [qk(B, H, K) for K in range(8, 33)]
            assert sizes == sorted(sizes), (B, H)
            if B >= 1000:
                assert qk(B, H, 9) > q(B, H) and qk(B, H, 32) - q(B, H) >= 4 * B * (32 - 8) - 256     # ds: B * K floats
    assert qk(10, 16, 0) == -1 and qk(10, 16, 33) == -1 and qk(-1, 16, 9) == -1


# ------------------------------------------------------------------------------ GPU --
def _adjudicated(got, ref32, ref64, what, mag):
    """ours against fp64 within the bar, or within 8x the fp32 reference's own worst error on that tensor"""
    got, ref32, ref64 = got.detach().cpu().double(), ref32.detach().double(), ref64.detach()
    atol = ATOL * max(1.0, mag)
    e_g64, e_r64 = (got - ref64).abs(), (ref32 - ref64).abs()
    fine = (e_g64 <= atol + RTOL * ref64.abs()) | (e_g64 <= 8.0 * float(e_r64.max()))
    assert bool(fine.all()), f"{what}: ours vs fp64 {float(e_g64.max()):.3e}, fp32 reference vs fp64 {float(e_r64.max()):.3e}"


def _check_against_oracle(cent, pos, emb, up, K, dev, oracle_dev="cpu"):
    """ctx, d_emb and the four MLP gradients of our module against the oracle in fp32 and fp64 (on `oracle_dev`);
    vehicles whose K-th and (K+1)-th distances are within 1e-6 relative are masked out of the upstream gradient"""
    import sldm_gnn_b200 as sg
    torch.manual_seed(5)
    orc = MapSpatialAttentionOracle(cent, K).to(oracle_dev)
    m = sg.MapSpatialAttention(cent, K).to(dev)
    m.load_state_dict(orc.state_dict(), strict=True)
    pos_o, emb_o, up_o = pos.to(oracle_dev), emb.to(oracle_dev), up.to(oracle_dev)
    ok = _mask_clear(orc, pos_o).to(oracle_dev)
    assert float(ok.float().mean()) > 0.9
    upm = up_o * ok[:, None]
    e_r = emb_o.clone().requires_grad_(True)
    o_r = orc(pos_o, e_r)
    (o_r * upm).sum().backward()
    o64 = MapSpatialAttentionOracle(cent.double(), K).double().to(oracle_dev)
    o64.load_state_dict({k: v.double() for k, v in orc.state_dict().items()})
    e_d = emb_o.double().requires_grad_(True)
    o_d = o64(pos_o.double(), e_d)
    (o_d * upm.double()).sum().backward()
    e_g = emb.to(dev).requires_grad_(True)
    o_g = m(pos.to(dev), e_g)
    (o_g * upm.to(dev)).sum().backward()
    okc = ok.cpu()
    _adjudicated(o_g[okc.to(dev)], o_r[ok].cpu(), o_d[ok].cpu(), "ctx", 1.0)
    _adjudicated(e_g.grad, e_r.grad.cpu(), e_d.grad.cpu(), "demb", float(e_d.grad.abs().max()))
    rp, dp = dict(orc.named_parameters()), dict(o64.named_parameters())
    mag = max(float(v.grad.abs().max()) for v in dp.values())
    for k, p in m.named_parameters():
        _adjudicated(p.grad, rp[k].grad.cpu(), dp[k].grad.cpu(), "grad " + k, mag)
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("B,S,D,K", [(1, 9, 8, 9), (257, 12, 32, 12), (77, 32, 7, 32), (9, 40, 7, 31), (1000, 3000, 32, 16),
                                     (64, 2049, 128, 32), (300, 5000, 16, 16), (50, 9000, 32, 32), (1003, 500, 40, 31),
                                     # busy segments: every segment is selected by hundreds of vehicles
                                     (2000, 40, 16, 32), (3000, 33, 8, 32), (1500, 60, 40, 9), (999, 20, 128, 16)])
def test_cuda_matches_oracle_random(B, S, D, K):
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(B + S + K)
    cent = torch.rand(S, 2, generator=g) * 500 - 250
    pos = torch.rand(B, 2, generator=g) * 500 - 250
    emb = torch.randn(S, D, generator=g)
    up = torch.randn(B, D, generator=g)
    m = _check_against_oracle(cent, pos, emb, up, K, dev)
    pos_g, emb_g = pos.to(dev), emb.to(dev)
    assert torch.equal(m(pos_g, emb_g), m(pos_g, emb_g))


@pytest.mark.gpu
def test_bench_scale_against_the_reference_op_chain_on_the_gpu():
    """The C2 step's vehicles at 1024 graphs, a 2048-segment map, D = 32, K = 32; the oracle runs on the GPU"""
    dev = torch.device("cuda:0")
    B, S, D, K = 205587, 2048, 32, 32
    g = torch.Generator().manual_seed(11)
    cent = torch.rand(S, 2, generator=g) * 2000
    pos = torch.rand(B, 2, generator=g) * 2000
    emb = torch.randn(S, D, generator=g)
    up = torch.randn(B, D, generator=g)
    _check_against_oracle(cent, pos, emb, up, K, dev, oracle_dev=dev)


def _wide_geometries():
    cases = {k: v for k, v in _geometries().items() if k not in ("S_equals_K", "single")}
    g = torch.Generator().manual_seed(78)
    cases["S_equals_32"] = (torch.rand(32, 2, generator=g), torch.rand(64, 2, generator=g) * 3 - 1, None)
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("K", [16, 32])
@pytest.mark.parametrize("name", list(_wide_geometries().keys()))
def test_grid_search_equals_exhaustive_scan(name, K):
    """Same (distance, index) keys, same epilogue: idx, dist, w and ctx are bit-identical"""
    dev = torch.device("cuda:0")
    cent, pos, _ = _wide_geometries()[name]
    S, D = cent.size(0), 16
    assert S >= K
    g = torch.Generator().manual_seed(S + K)
    emb = torch.randn(S, D, generator=g).to(dev)
    params = [t.to(dev) for t in (torch.randn(16, generator=g), torch.randn(16, generator=g), torch.randn(16, generator=g),
                                  torch.randn(1, generator=g))]
    cent, pos = cent.to(dev).contiguous(), pos.to(dev).contiguous()
    a = _forward_raw("scan", pos, cent, emb, params, K)
    b = _forward_raw("grid", pos, cent, emb, params, K)
    for x, y, what in zip(a, b, ("idx", "dist", "w", "ctx")):
        assert torch.equal(x, y), f"{name}: {what} differs in {int((x != y).sum())} places"
    idx, dist = b[0], b[1]
    assert bool((dist[:, 1:] >= dist[:, :-1]).all())
    same = dist[:, 1:] == dist[:, :-1]
    assert bool((idx[:, 1:][same] > idx[:, :-1][same]).all())
    assert bool((idx >= 0).all()) and bool((idx < S).all())
    if S <= 20000:
        full = torch.cdist(pos.double(), cent.double())
        kth = full.gather(1, idx[:, -1:])
        assert int(((full < kth * (1 - 1e-6)).sum(1) > K - 1).sum()) == 0
    if name == "identical":                         # all distances equal: the K lowest indices, in order
        assert torch.equal(idx, torch.arange(K, device=dev).expand_as(idx))


_NAME = re.compile(r"(k_map_\w+)(<[^>]*>)?")


def _map_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        m = _NAME.search(e.name)
        if m and e.device_type == torch.autograd.DeviceType.CUDA:
            names.add(m.group(1) + (m.group(2) or "").replace(" ", ""))
    return names


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 5, 8, 9, 32])
def test_launches_by_k(K, monkeypatch):
    """K <= 8 runs exactly the kernels it ran before this path existed; K > 8 runs the warp-per-vehicle kernels"""
    import sldm_gnn_b200 as sg
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(K)
    S, B = 300, 1000
    cent = torch.rand(S, 2, generator=g) * 100
    m = sg.MapSpatialAttention(cent, K).to(dev)
    pos = (torch.rand(B, 2, generator=g) * 100).to(dev)
    for D, vec in ((16, True), (7, False)):
        emb = torch.randn(S, D, generator=g).to(dev).requires_grad_(True)
        for scan in (False, True):
            if scan:
                monkeypatch.setenv("SLDM_MAP_ATTENTION_SCAN", "1")
            else:
                monkeypatch.delenv("SLDM_MAP_ATTENTION_SCAN", raising=False)
            m(pos, emb)                             # the grid is built outside the recorded window
            out = {}
            fwd = _map_kernels(lambda: out.setdefault("y", m(pos, emb)))
            bwd = _map_kernels(lambda: out["y"].sum().backward())
            if K <= 8:
                want_f = {f"k_map_attention_fwd<{K}>" if scan else f"k_map_attention_grid_fwd<{K}>"}
                want_b = {f"k_map_attention_bwd_ds<{K},{8 if vec else 32}>", "k_map_attention_bwd_mlp", "k_map_attention_reduce",
                          f"k_map_attention_demb<{K}>"}
            else:
                want_f = {"k_map_attention_fwd_wide" if scan else "k_map_attention_grid_fwd_wide"}
                want_b = {f"k_map_attention_bwd_ds_wide<{'true' if vec else 'false'}>", "k_map_attention_bwd_mlp_wide",
                          "k_map_attention_reduce", f"k_map_attention_demb<{K}>"}
            assert fwd == want_f, (K, D, scan, fwd)
            assert bwd == want_b, (K, D, scan, bwd)


@pytest.mark.gpu
def test_edge_cases():
    import sldm_gnn_b200 as sg
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(1)
    cent = torch.rand(40, 2, generator=g) * 10
    m = sg.MapSpatialAttention(cent, 16).to(dev)
    emb = torch.randn(40, 8, generator=g).to(dev).requires_grad_(True)
    out = m(torch.empty(0, 2, device=dev), emb)
    assert out.shape == (0, 8)
    out.sum().backward()
    assert torch.equal(emb.grad, torch.zeros_like(emb)) and all(bool((p.grad == 0).all()) for p in m.parameters())
    pos = (torch.rand(37, 2, generator=g) * 10).to(dev)
    with torch.inference_mode():
        got = m(pos, emb.detach())
        assert got.shape == (37, 8)
    assert torch.equal(got, m(pos, emb).detach())
    # K = S = 32: every segment is selected, the weights a softmax over all of them
    c32 = torch.rand(32, 2, generator=g)
    m32 = sg.MapSpatialAttention(c32, 32).to(dev)
    e32 = torch.randn(32, 4, generator=g)
    p32 = torch.rand(50, 2, generator=g)
    _check_against_oracle(c32, p32, e32, torch.randn(50, 4, generator=g), 32, dev)
    assert m32(p32.to(dev), e32.to(dev)).shape == (50, 4)
    with pytest.raises(NotImplementedError, match="32"):
        sg.MapSpatialAttention(torch.rand(40, 2), 33).to(dev)(torch.rand(3, 2, device=dev), torch.randn(40, 8, device=dev))
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        sg.MapSpatialAttention(torch.rand(10, 2), 20).to(dev)(torch.rand(3, 2, device=dev), torch.randn(10, 8, device=dev))


@pytest.mark.gpu
def test_forward_and_gradients_are_deterministic():
    import sldm_gnn_b200 as sg
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(2)
    S = 2048
    m = sg.MapSpatialAttention(torch.rand(S, 2, generator=g) * 2000, 32).to(dev)
    pos = torch.cat([torch.rand(20000, 2, generator=g) * 2000, torch.zeros(3000, 2)]).to(dev)   # plus one busy spot
    emb = torch.randn(S, 32, generator=g).to(dev)
    up = torch.randn(pos.size(0), 32, generator=g).to(dev)

    def run():
        m.zero_grad(set_to_none=True)
        e = emb.clone().requires_grad_(True)
        y = m(pos, e)
        (y * up).sum().backward()
        return [y.detach(), e.grad] + [p.grad.clone() for p in m.parameters()]

    a, b = run(), run()
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# ------------------------------------------------------------------------------ the model --
@pytest.mark.gpu
@pytest.mark.parametrize("path", GRUSAGE_GOLDEN, ids=lambda p: p.rsplit("/", 1)[-1])
def test_cuda_model_with_top16_matches_the_oracle_composition(path):
    """The golden model configurations (map_tensors and map_embeddings modes) with map_attention_topk = 16, against the
    oracle composition: fp32 and fp64 on the CPU, and fp32 on the GPU's library kernels (cuDNN off) for the noise floor"""
    import sldm_gnn_b200 as sg
    dev = torch.device("cuda:0")
    fx = torch.load(path, weights_only=False)
    fx["kwargs"] = dict(fx["kwargs"], map_attention_topk=16)
    model = _build(sg.GruSage, fx, dev)
    logits, loss, grads = _step(model, fx, dev)
    ref_logits, ref_loss, ref_grads = _step(_build(GruSageOracle, fx), fx)
    with torch.backends.cudnn.flags(enabled=False):
        lib_logits, lib_loss, lib_grads = _step(_build(GruSageOracle, fx, dev), fx, dev)
    to64 = lambda v: v.double() if isinstance(v, torch.Tensor) and v.is_floating_point() else v
    fx64 = dict(fx, state_dict={k: to64(v) for k, v in fx["state_dict"].items()}, map={k: to64(v) for k, v in fx["map"].items()},
                extra_emb=to64(fx["extra_emb"]), data={k: to64(v) for k, v in fx["data"].items()})
    m64 = _build(GruSageOracle, fx64).double()
    data64 = Bag(fx64["data"])
    l64 = m64(data64)
    loss64 = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(fx["pos_weight"], dtype=torch.float64))(l64, data64.y)
    loss64.backward()
    grads64 = {k: p.grad for k, p in m64.named_parameters()}

    def adjudicated(got, ref32, lib32, ref64, what):
        got, ref32, lib32, ref64 = got.cpu().double(), ref32.double(), lib32.cpu().double(), ref64.detach()
        mag = max(1.0, float(ref64.abs().max()))
        e_g = (got - ref64).abs()
        floor = max(float((ref32 - ref64).abs().max()), float((lib32 - ref64).abs().max()))
        fine = (e_g <= ATOL * mag + RTOL * ref64.abs()) | (e_g <= 8.0 * floor)
        assert bool(fine.all()), f"{what}: ours vs fp64 {float(e_g.max()):.3e}, fp32 noise floor {floor:.3e}"

    adjudicated(logits, ref_logits, lib_logits, l64, "logits")
    adjudicated(loss, ref_loss, lib_loss, loss64, "loss")
    assert set(grads) == set(grads64)
    for k in grads:
        adjudicated(grads[k], ref_grads[k], lib_grads[k], grads64[k], "grad " + k)


def _c2_like_top16(dev, seed=0):
    """test_grusage's small full model (map encoder + attention + GRU head, a 48-segment map) with map_attention_topk = 16,
    and its batch builder.  The padding rows of the graphed wrappers all select the same 16 segments."""
    from types import SimpleNamespace
    import sldm_gnn_b200 as sg
    g = torch.Generator().manual_seed(100 + seed)
    S = 48
    mt = dict(float_features=torch.randn(S, 6, generator=g), bool_features=torch.rand(S, 3, generator=g) > 0.5,
              lane_type_cats=torch.randint(0, 4, (S,), generator=g),
              mgraph_edge_indexes=torch.stack([torch.randint(0, S, (4 * S,), generator=g), torch.randint(0, S, (4 * S,), generator=g)]),
              mseg_centroids=torch.rand(S, 2, generator=g) * 100.0)
    kw = dict(dynamic_features_num=6, frames_num=8, gru_hidden_size=32, gru_num_layers=1, fc1dims=[24], sage_hidden_dims=[32, 32],
              fc2dims=[16], out_dim=1, num_st_types=9, emb_dim=4, dropout=None, negative_slope=0.1, global_pooling="double",
              mapenc_lane_embdim=4, mapenc_sage_hdims=[16, 16], map_attention_topk=16)
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
def test_graphed_grusage_with_top16_matches_the_uncaptured_model():
    from sldm_gnn_b200.grusage import GraphedGruSage
    dev = torch.device("cuda:0")
    model, batch = _c2_like_top16(dev)
    assert model.map_attention.k == 16
    crit = torch.nn.BCEWithLogitsLoss()
    g = GraphedGruSage(model, max_nodes=128, max_edges=512, max_graphs=12, training=True)
    for graphs, seed in ((11, 1), (5, 2), (8, 3)):
        data = batch(graphs, seed)
        model.zero_grad(set_to_none=True)
        ref_logits = model(data)
        crit(ref_logits, data.y).backward()
        ref = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
        model.zero_grad(set_to_none=True)
        out = g(data)
        assert torch.allclose(out, ref_logits, rtol=1e-5, atol=1e-6), float((out - ref_logits).abs().max())
        crit(out, data.y).backward()
        got = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}
        assert set(got) == set(ref) and "map_attention.attn_mlp.0.weight" in got
        for k in ref:
            scale = max(1.0, float(ref[k].abs().max()))
            assert torch.allclose(got[k], ref[k], rtol=1e-4, atol=2e-6 * scale), (k, float((got[k] - ref[k]).abs().max()))
    model.eval()
    data = batch(6, 7)
    with torch.inference_mode():
        want = model(data)
    gi = GraphedGruSage(model, max_nodes=96, max_edges=400, max_graphs=8, training=False)
    got = gi(data)
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-6), float((got - want).abs().max())


@pytest.mark.gpu
def test_graphed_train_step_with_top16_follows_the_eager_loop():
    import torch.nn.functional as Fn
    from sldm_gnn_b200.grusage import GraphedTrainStep
    dev = torch.device("cuda:0")
    model, batch = _c2_like_top16(dev, seed=2)
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
        opt_g.zero_grad(set_to_none=True)
        lg = step(data, data.y)
        if i == 0:
            ge = dict(twin.named_parameters())
            for k, p in model.named_parameters():
                scale = max(1.0, float(ge[k].grad.abs().max()))
                assert torch.allclose(p.grad, ge[k].grad, rtol=1e-4, atol=2e-6 * scale), (k, float((p.grad - ge[k].grad).abs().max()))
        opt_e.step()
        losses_e.append(float(le)); losses_g.append(float(lg))
    assert all(abs(a - b) <= 2e-3 * max(1.0, abs(a)) for a, b in zip(losses_e, losses_g)), (losses_e, losses_g)
