"""MapSpatialAttention (SURVEY 8f rank 3; src/models/map/mapattention.py:5-56).

Parity is PINNED here: the reference class is plain torch, so the golden vectors under tests/golden/map_attention were
produced by the reference itself, and the oracle restatement reproduces them bit for bit.  Tolerance: rtol 1e-5 /
atol 1e-6 on the context vectors and the gradients (the MLP, softmax and the weighted sum are fp32 with a different association than ATen's), adjudicated against an fp64 run of
the oracle where the fp32 reference itself is no more accurate than that; neighbour indices and distances exact
except for vehicles whose K-th and (K+1)-th distances are closer than 1e-6 relative (the order of near ties is
unspecified in torch.topk), which are skipped."""
import glob
import os

import pytest
import torch

from oracle.map_attention_oracle import MapSpatialAttentionOracle

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "map_attention", "*.pt")))
RTOL, ATOL = 1e-5, 1e-6


def _close(a, b, what, scale=False, scale_ref=None):
    """scale_ref: parameter gradients are sums of the same B*K terms; d(bias of the last layer) = sum_k ds_k is exactly 0
    in exact arithmetic (softmax backward), so its rounding noise is measured against the magnitude of its sibling
    gradients, not against its own (zero) value."""
    a, b = a.detach().cpu(), b.detach().cpu()
    ref_mag = float(b.abs().max()) if scale_ref is None else scale_ref
    atol = ATOL * (max(1.0, ref_mag) if (scale or scale_ref is not None) else 1.0)
    err = (a - b).abs()
    assert bool((err <= atol + RTOL * b.abs()).all()), f"{what}: max err {float(err.max()):.3e}"


# ------------------------------------------------------------------------------ CPU --
def test_golden_files_exist():
    assert len(GOLDEN) == 4


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_oracle_reproduces_reference_golden(path):
    d = torch.load(path)
    m = MapSpatialAttentionOracle(d["centroids"], d["k"])
    m.load_state_dict(d["state_dict"], strict=True)
    emb = d["emb"].clone().requires_grad_(True)
    out = m(d["pos"], emb)
    (out * d["upstream"]).sum().backward()
    assert torch.equal(out.detach(), d["out"])                      # same torch ops, same machine class: bit equal
    assert torch.allclose(emb.grad, d["demb"], rtol=1e-6, atol=1e-7)
    for k, p in m.named_parameters():
        assert torch.allclose(p.grad, d["dparams"][k], rtol=1e-6, atol=1e-7), k


def test_module_contract_matches_reference_fixture():
    import sldm_gnn_b200 as sg
    d = torch.load(GOLDEN[0])
    m = sg.MapSpatialAttention(d["centroids"], d["k"])
    m.load_state_dict(d["state_dict"], strict=True)                 # same keys, same shapes
    assert "map_centroids" not in m.state_dict()                    # non-persistent buffer, like the reference
    with pytest.raises(RuntimeError):
        m(d["pos"], d["emb"])                                       # CPU tensors: no fallback


# ------------------------------------------------------------------------------ GPU --
def _mask_clear(orc, pos):
    """vehicles whose K-th and (K+1)-th nearest distances are clearly separated"""
    d, _ = orc.neighbours(pos)
    if d.size(1) <= orc.k:
        return torch.ones(pos.size(0), dtype=torch.bool)
    a, b = d[:, orc.k - 1], d[:, orc.k]
    return (b - a) > 1e-6 * b.abs().clamp(min=1e-30)


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_cuda_matches_reference_golden(path):
    import sldm_gnn_b200 as sg
    dev = torch.device("cuda:0")
    d = torch.load(path)
    m = sg.MapSpatialAttention(d["centroids"], d["k"]).to(dev)
    m.load_state_dict(d["state_dict"], strict=True)
    emb = d["emb"].to(dev).requires_grad_(True)
    out = m(d["pos"].to(dev), emb)
    (out * d["upstream"].to(dev)).sum().backward()
    orc = MapSpatialAttentionOracle(d["centroids"], d["k"])
    ok = _mask_clear(orc, d["pos"])
    assert float(ok.float().mean()) > 0.95
    _close(out[ok.to(dev)], d["out"][ok], "ctx")
    if bool(ok.all()):
        _close(emb.grad, d["demb"], "demb", scale=True)
        mag = 10.0 * max(float(v.abs().max()) for v in d["dparams"].values())
        for k, p in m.named_parameters():
            _close(p.grad, d["dparams"][k], "grad " + k, scale_ref=mag)


@pytest.mark.gpu
@pytest.mark.parametrize("B,S,D,K", [(1, 5, 4, 5), (257, 33, 32, 5), (1000, 3000, 32, 5), (64, 2049, 128, 8), (9, 40, 7, 2),
                                     (300, 5000, 16, 5), (50, 9000, 32, 3),    # more than 4096 segments: tiled scan
                                     # busy segments (>= 32 selecting positions each) with an embedding width that leaves
                                     # lanes idle in k_map_attention_demb: D = 8 is the reference's default map width
                                     (2000, 12, 16, 3), (3000, 7, 8, 5), (1500, 20, 40, 4)])
def test_cuda_matches_oracle_random(B, S, D, K):
    import sldm_gnn_b200 as sg
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(B + S)
    cent = torch.rand(S, 2, generator=g) * 500 - 250
    pos = torch.rand(B, 2, generator=g) * 500 - 250
    emb = torch.randn(S, D, generator=g)
    up = torch.randn(B, D, generator=g)
    torch.manual_seed(5)
    orc = MapSpatialAttentionOracle(cent, K)
    m = sg.MapSpatialAttention(cent, K).to(dev)
    m.load_state_dict(orc.state_dict(), strict=True)
    ok = _mask_clear(orc, pos)
    e_r = emb.clone().requires_grad_(True)
    o_r = orc(pos, e_r)
    (o_r * up * ok[:, None]).sum().backward()
    # fp64 adjudicator: the softmax backward (w * (g - <w,g>)) cancels, so the fp32 reference itself is only accurate
    # to a few 1e-5 relative on the MLP gradients of small batches; our error against the exact answer must stay within
    # the bar or within 8x the fp32 reference's own worst error on that tensor (same order of magnitude: the two fp32
    # evaluations differ in the association of the dot products / MLP / softmax sums and in expf vs ATen's exp, and the
    # ratio of two independent draws of rounding noise over a 16-element tensor reaches 4-5 in these cases)
    o64 = MapSpatialAttentionOracle(cent.double(), K).double()
    o64.load_state_dict({k: v.double() for k, v in orc.state_dict().items()})
    e_d = emb.double().requires_grad_(True)
    o_d = o64(pos.double(), e_d)
    (o_d * (up * ok[:, None]).double()).sum().backward()
    e_g = emb.to(dev).requires_grad_(True)
    o_g = m(pos.to(dev), e_g)
    (o_g * (up * ok[:, None]).to(dev)).sum().backward()

    def adjudicated(got, ref32, ref64, what, mag):
        got, ref32, ref64 = got.detach().cpu().double(), ref32.detach().double(), ref64.detach()
        atol = ATOL * max(1.0, mag)
        e_g64, e_r64 = (got - ref64).abs(), (ref32 - ref64).abs()
        fine = (e_g64 <= atol + RTOL * ref64.abs()) | (e_g64 <= 8.0 * float(e_r64.max()))
        assert bool(fine.all()), f"{what}: ours vs fp64 {float(e_g64.max()):.3e}, fp32 reference vs fp64 {float(e_r64.max()):.3e}"

    # the scores are MLP(distance) with distances of a few hundred: an fp32 rounding of the score (1e-5 absolute) moves the
    # softmax weights by 1e-5 relative in the fp32 reference as well, so the context vectors are adjudicated too
    adjudicated(o_g[ok.to(dev)], o_r[ok], o_d[ok], "ctx", 1.0)
    adjudicated(e_g.grad, e_r.grad, e_d.grad, "demb", float(e_d.grad.abs().max()))
    rp, dp = dict(orc.named_parameters()), dict(o64.named_parameters())
    mag = max(float(v.grad.abs().max()) for v in dp.values())
    for k, p in m.named_parameters():
        adjudicated(p.grad, rp[k].grad, dp[k].grad, "grad " + k, mag)
    # determinism
    assert torch.equal(m(pos.to(dev), emb.to(dev)), m(pos.to(dev), emb.to(dev)))


@pytest.mark.gpu
def test_cuda_edge_cases_and_modes():
    import sldm_gnn_b200 as sg
    dev = torch.device("cuda:0")
    cent = torch.randn(10, 2)
    m = sg.MapSpatialAttention(cent, 5).to(dev)
    out = m(torch.empty(0, 2, device=dev), torch.randn(10, 8, device=dev))
    assert out.shape == (0, 8)
    with torch.inference_mode():
        assert m(torch.randn(3, 2, device=dev), torch.randn(10, 8, device=dev)).shape == (3, 8)
    with pytest.raises(RuntimeError):
        sg.MapSpatialAttention(torch.randn(3, 2), 5).to(dev)(torch.randn(2, 2, device=dev), torch.randn(3, 8, device=dev))
    # duplicate centroids: ties go to the lower index, the result is still a valid convex combination
    cent2 = torch.zeros(6, 2)
    m2 = sg.MapSpatialAttention(cent2, 3).to(dev)
    emb = torch.arange(6.).view(6, 1).to(dev)
    o = m2(torch.ones(4, 2, device=dev), emb)
    assert torch.allclose(o, torch.full((4, 1), 1.0, device=dev))     # equal distances -> equal weights over segments 0,1,2


# ------------------------------------------------------------------ grid search vs exhaustive scan --
def _forward_raw(kind, pos, cent, emb, params, K):
    """idx / dist / w / ctx of one forward straight through the C-ABI; kind = 'scan' | 'grid'."""
    from sldm_gnn_b200._lib import lib, check
    dev = pos.device
    B, S, D, H = pos.size(0), cent.size(0), emb.size(1), params[0].numel()
    ctx = torch.empty(B, D, device=dev)
    idx = torch.empty(B, K, dtype=torch.long, device=dev)
    dist, w = torch.empty(B, K, device=dev), torch.empty(B, K, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    W1, b1, W2, b2 = params
    if kind == "scan":
        check(lib.sldm_map_attention_forward(pos.data_ptr(), B, cent.data_ptr(), S, emb.data_ptr(), D, K, W1.data_ptr(), b1.data_ptr(),
                                             W2.data_ptr(), b2.data_ptr(), H, ctx.data_ptr(), idx.data_ptr(), dist.data_ptr(), w.data_ptr(), st))
    else:
        nb = int(lib.sldm_map_grid_bytes(S))
        grid = torch.empty(nb, dtype=torch.uint8, device=dev)
        check(lib.sldm_map_grid_build(cent.data_ptr(), S, grid.data_ptr(), nb, st))
        check(lib.sldm_map_attention_forward_grid(pos.data_ptr(), B, grid.data_ptr(), nb, S, emb.data_ptr(), D, K, W1.data_ptr(),
                                                  b1.data_ptr(), W2.data_ptr(), b2.data_ptr(), H, ctx.data_ptr(), idx.data_ptr(),
                                                  dist.data_ptr(), w.data_ptr(), st))
    torch.cuda.synchronize()
    return idx, dist, w, ctx


def _geometries():
    g = torch.Generator().manual_seed(77)
    r = lambda *s: torch.rand(*s, generator=g)
    lattice = torch.stack(torch.meshgrid(torch.arange(40.), torch.arange(30.), indexing="ij"), -1).reshape(-1, 2)
    clusters = (torch.randint(0, 6, (3000, 1), generator=g).float() * 400.0) + torch.randn(3000, 2, generator=g) * 0.5
    cases = {
        "uniform": (r(2048, 2) * 2000, r(5000, 2) * 2000, 5),
        "outside": (r(1500, 2) * 100, torch.cat([r(2000, 2) * 3000 - 1500, torch.tensor([[0., 0.], [100., 100.], [-1e6, 50.], [50., 1e7]])]), 5),
        "clustered": (clusters, torch.cat([clusters[:500] + 0.1, r(1500, 2) * 2400 - 200]), 8),
        "collinear_x": (torch.stack([r(700) * 50, torch.full((700,), 3.25)], 1), r(900, 2) * 60 - 5, 4),
        "collinear_y": (torch.stack([torch.full((700,), -7.5), r(700) * 50], 1), r(900, 2) * 60 - 5, 4),
        "identical": (torch.full((300, 2), 12.5), r(100, 2) * 30, 6),
        "lattice_ties": (lattice, torch.cat([lattice[::7], lattice[::5] + 0.5, lattice[::3] + torch.tensor([0.5, 0.0])]), 5),
        "on_centroids": (r(999, 2) * 10, (r(999, 2) * 10)[:0].new_zeros(0, 2), 3),      # positions filled in below
        "S_equals_K": (r(5, 2), r(64, 2) * 3 - 1, 5),
        "single": (r(1, 2), r(33, 2), 1),
        "far_offset": (r(4000, 2) * 300 + 1.0e6, r(3000, 2) * 320 + 1.0e6 - 10, 5),     # ulp of the coordinates = 0.06
        "tiny_extent": (r(2000, 2) * 1e-3, r(1000, 2) * 1.2e-3, 5),
        "large_map": (r(20000, 2) * 5000, r(4000, 2) * 5000, 5),
        "grid_side_cap": (r(1200000, 2) * 9000, r(600, 2) * 9000, 5),                    # G capped at 512
    }
    c, _, k = cases["on_centroids"]
    cases["on_centroids"] = (c, c.clone(), k)
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(_geometries().keys()))
def test_grid_search_equals_exhaustive_scan(name):
    """Same (distance, index) keys, same arithmetic after the selection: every output is bit-identical."""
    dev = torch.device("cuda:0")
    cent, pos, K = _geometries()[name]
    S, D = cent.size(0), 16
    g = torch.Generator().manual_seed(S)
    emb = torch.randn(S, D, generator=g).to(dev)
    params = [t.to(dev) for t in (torch.randn(16, generator=g), torch.randn(16, generator=g), torch.randn(16, generator=g),
                                  torch.randn(1, generator=g))]
    cent, pos = cent.to(dev).contiguous(), pos.to(dev).contiguous()
    a = _forward_raw("scan", pos, cent, emb, params, K)
    b = _forward_raw("grid", pos, cent, emb, params, K)
    for x, y, what in zip(a, b, ("idx", "dist", "w", "ctx")):
        assert torch.equal(x, y), f"{name}: {what} differs in {int((x != y).sum())} places"
    # and the selection is the true K nearest: distances ascending, ties by index, nothing closer left out
    idx, dist = b[0], b[1]
    assert bool((dist[:, 1:] >= dist[:, :-1]).all())
    same = dist[:, 1:] == dist[:, :-1]
    assert bool((idx[:, 1:][same] > idx[:, :-1][same]).all())
    if S <= 20000:
        full = torch.cdist(pos.double(), cent.double())
        kth = full.gather(1, idx[:, -1:])
        assert int(((full < kth * (1 - 1e-6)).sum(1) > K - 1).sum()) == 0


@pytest.mark.gpu
def test_grid_follows_the_centroid_buffer(monkeypatch):
    import sldm_gnn_b200 as sg
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(3)
    cent = torch.rand(500, 2, generator=g) * 100
    m = sg.MapSpatialAttention(cent, 5).to(dev)
    pos, emb = (torch.rand(300, 2, generator=g) * 100).to(dev), torch.randn(500, 8, generator=g).to(dev)
    o1 = m(pos, emb)
    grid1 = m._grid
    assert m(pos, emb) is not None and m._grid is grid1                      # cached
    m.map_centroids.copy_(torch.rand(500, 2, generator=g).to(dev) * 100)     # in-place write -> rebuilt
    o2 = m(pos, emb)
    assert m._grid is not grid1 and not torch.equal(o1, o2)
    monkeypatch.setenv("SLDM_MAP_ATTENTION_SCAN", "1")
    assert torch.equal(m(pos, emb), o2)
