"""Proximity edges for windows of any length (src/gbuilder.py:88-112, :244-268, rcv.py:77), compared for equality.

numpy sums float32 arrays of more than 128 elements by recursive halving (numpy/_core/src/umath/loops_utils.h.src,
pairwise_sum), and `edge_build.cu` streams each pair's distances through that tree.  The CPU tests pin numpy's
arithmetic and check the kernel's leaf-and-stack schedule against the recursive tree; the GPU tests require
`edge_index` and all four `edge_attr` columns to equal the reference loop's (oracle/edges_oracle.py) bit for bit."""
import numpy as np
import pytest
import torch

from oracle.edges_oracle import proximity_edges_oracle

LEAF = 128


def _split(n):
    h = n // 2
    return h - h % 8


def np_pairwise_sum(a):
    """numpy's float32 pairwise sum of a 1-D float32 array, restated."""
    def pw(lo, n):
        if n < 8:
            r = np.float32(0)
            for k in range(n):
                r = np.float32(r + a[lo + k])
            return r
        if n <= LEAF:
            r = [np.float32(a[lo + k]) for k in range(8)]
            i = 8
            while i < n - n % 8:
                for k in range(8):
                    r[k] = np.float32(r[k] + a[lo + i + k])
                i += 8
            res = np.float32(np.float32(np.float32(r[0] + r[1]) + np.float32(r[2] + r[3]))
                             + np.float32(np.float32(r[4] + r[5]) + np.float32(r[6] + r[7])))
            for k in range(i, n):
                res = np.float32(res + a[lo + k])
            return res
        n2 = _split(n)
        return np.float32(pw(lo, n2) + pw(lo + n2, n - n2))
    return pw(0, len(a))


def np_mean(a):
    return np.float32(np_pairwise_sum(a) / np.float32(len(a)))


def _recursive_tree(n):
    """numpy's addition tree over elements 0..n-1 as nested ('+', l, r) tuples."""
    def pw(lo, n):
        if n < 8:
            t = 0
            for k in range(n):
                t = ("+", t, lo + k)
            return t
        if n <= LEAF:
            r = [lo + k for k in range(8)]
            i = 8
            while i < n - n % 8:
                r = [("+", r[k], lo + i + k) for k in range(8)]
                i += 8
            t = ("+", ("+", ("+", r[0], r[1]), ("+", r[2], r[3])), ("+", ("+", r[4], r[5]), ("+", r[6], r[7])))
            for k in range(i, n):
                t = ("+", t, lo + k)
            return t
        n2 = _split(n)
        return ("+", pw(lo, n2), pw(lo + n2, n - n2))
    return pw(0, n)


def _streamed_tree(n, stack_depth=25):
    """The schedule of `pair_sums` in edge_build.cu, step for step: leaves summed as elements arrive (running sums start
    at 0), finished leaves combined in post-order through a fixed-depth stack of left halves, the parent's size
    recomputed from the root along the path bits."""
    stk = [None] * stack_depth
    right, depth, m, nxt = 0, 0, n, 0
    while True:
        while m > LEAF:
            m = _split(m)
            depth += 1
        r = [0] * 8
        for _ in range(m >> 3):
            for k in range(8):
                r[k] = ("+", r[k], nxt)
                nxt += 1
        s = ("+", ("+", ("+", r[0], r[1]), ("+", r[2], r[3])), ("+", ("+", r[4], r[5]), ("+", r[6], r[7])))
        for _ in range(m & 7):
            s = ("+", s, nxt)
            nxt += 1
        while depth > 0 and (right >> (depth - 1)) & 1:
            depth -= 1
            right &= ~(1 << depth)
            s = ("+", stk[depth], s)
        if depth == 0:
            break
        stk[depth - 1] = s
        right |= 1 << (depth - 1)
        p = n
        for lvl in range(depth - 1):
            h = _split(p)
            p = p - h if (right >> lvl) & 1 else h
        m = p - _split(p)
    assert nxt == n
    return s


def _drop_zero(t):
    """0 + a == a for the non-negative distances: remove additions of the literal 0 a running sum starts from."""
    if not isinstance(t, tuple):
        return t
    l, r = _drop_zero(t[1]), _drop_zero(t[2])
    if l == 0:
        return r
    if r == 0:
        return l
    return ("+", l, r)


def test_pairwise_sum_restatement_matches_numpy():
    rng = np.random.default_rng(0)
    sizes = list(range(0, 1101)) + [2047, 4096, 4097, 5000, 9000, 20000]
    for n in sizes:
        a = (rng.random(n, dtype=np.float32) * rng.choice([1.0, 100.0, 1e4])).astype(np.float32)
        got = np_pairwise_sum(a)
        assert got.dtype == np.float32 and got.tobytes() == np.add.reduce(a).tobytes(), n
        if n:
            assert np_mean(a).tobytes() == a.mean().tobytes(), n
            sq = a ** 2
            assert np_mean(sq).tobytes() == sq.mean().tobytes(), n


def test_streamed_schedule_is_numpys_tree():
    for n in range(1, 4097):
        assert _drop_zero(_streamed_tree(n)) == _drop_zero(_recursive_tree(n)), n


def test_stack_depth_covers_int32_frame_counts():
    def right_path(n):                                       # how kEbStack is computed in edge_build.cu
        d = 0
        while n > LEAF:
            n -= _split(n)
            d += 1
        return d

    def deepest(n):
        return 0 if n <= LEAF else 1 + max(deepest(_split(n)), deepest(n - _split(n)))

    assert right_path(2 ** 31 - 1) == 25                     # kEbStack
    for n in (129, 1000, 4097, 1 << 20, 3 << 20):            # the right half is never the shallower one
        assert deepest(n) == right_path(n)


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _traj(V, T, seed, spread=60.0, p_present=0.8):
    g = torch.Generator().manual_seed(seed)
    x = torch.zeros(V, T, 6)
    start = (torch.rand(V, 1, 2, generator=g) - 0.5) * spread
    vel = (torch.rand(V, 1, 2, generator=g) - 0.5) * 4.0
    x[:, :, :2] = start + vel * torch.arange(T).view(1, T, 1) + torch.randn(V, T, 2, generator=g)
    x[:, :, 2] = torch.rand(V, T, generator=g) * 30
    x[:, :, 3] = torch.rand(V, T, generator=g) * 6.28
    x[:, :, 4] = (torch.rand(V, T, generator=g) < p_present).float()
    x[:, :, 5] = torch.rand(V, T, generator=g)
    return x


def _check_equal(x, radius):
    import sldm_gnn_b200 as sg
    ei_r, ea_r = proximity_edges_oracle(x, radius)
    ei_g, ea_g = sg.build_proximity_edges(x.cuda(), radius)
    assert ei_g.dtype == torch.long and ea_g.dtype == torch.float32
    assert torch.equal(ei_g.cpu(), ei_r), f"edge lists differ: {tuple(ei_g.shape)} vs {tuple(ei_r.shape)}"
    for c, name in enumerate(("min", "max", "mean", "mean of squares")):
        got, want = ea_g[:, c].cpu(), ea_r[:, c]
        assert torch.equal(got, want), \
            f"{name}: {int((got != want).sum())} of {want.numel()} differ from numpy"
    return ei_r.size(1)


LONG_T = [129, 130, 136, 200, 256, 257, 263, 1000, 4096, 4097]
_V = {129: 300, 130: 97, 136: 64, 200: 150, 256: 33, 257: 1, 263: 41, 1000: 24, 4096: 12, 4097: 9}
_RADIUS = {"none": 0.0, "some": 6.0, "all": 1e9}


@pytest.mark.gpu
@pytest.mark.parametrize("pp", [1.0, 0.9, 0.5])
@pytest.mark.parametrize("T", LONG_T)
def test_long_windows_equal_the_reference_loop(T, pp):
    V = _V[T]
    for k, (name, r) in enumerate(_RADIUS.items()):
        x = _traj(V, T, seed=T * 7 + k, spread=40.0, p_present=pp)
        E = _check_equal(x, r)
        if name == "all" and V > 1 and pp > 0.5:
            assert E == V * (V - 1)                          # every pair shares frames, so every pair is an edge


@pytest.mark.gpu
@pytest.mark.parametrize("V,T", [(2, 300), (300, 140), (5, 20000)])
def test_every_vehicle_absent(V, T):
    x = _traj(V, T, seed=3, p_present=0.0)
    assert _check_equal(x, 1e9) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("pp", [1.0, 0.7])
def test_window_longer_than_shared_memory_could_stage(pp):
    # 24 000 frames x {X, Y, presence} x 4 bytes = 288 KB: more than one CTA's shared memory can hold
    x = _traj(5, 24000, seed=11, spread=30.0, p_present=pp)
    assert _check_equal(x, 25.0) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("V,T,radius,pp", [(40, 16, 15.0, 0.8), (1, 16, 5.0, 1.0), (7, 5, 1000.0, 1.0), (120, 16, 8.0, 0.5),
                                           (300, 20, 12.0, 0.9), (33, 9, 0.0, 1.0), (25, 16, 20.0, 0.0), (64, 128, 10.0, 0.7)])
def test_short_windows_equal_the_reference_loop(V, T, radius, pp):
    from test_edges import _traj as traj16
    _check_equal(traj16(V, T, seed=V + T, p_present=pp), radius)


@pytest.mark.gpu
def test_two_calls_give_identical_results():
    import sldm_gnn_b200 as sg
    x = _traj(200, 1500, seed=5, p_present=0.9).cuda()
    a = sg.build_proximity_edges(x, 10.0)
    b = sg.build_proximity_edges(x, 10.0)
    assert a[0].numel() > 0
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
def test_strided_input_and_extra_features():
    x = _traj(30, 300, seed=9, p_present=0.9)
    wide = torch.cat([x, torch.rand(30, 300, 3)], dim=2)    # F = 9: only X, Y and presence are read
    _check_equal(wide, 8.0)
    import sldm_gnn_b200 as sg
    xt = x.transpose(0, 1).contiguous().cuda().transpose(0, 1)
    ei, ea = sg.build_proximity_edges(xt, 8.0)
    ei_r, ea_r = proximity_edges_oracle(x, 8.0)
    assert torch.equal(ei.cpu(), ei_r) and torch.equal(ea.cpu(), ea_r)


@pytest.mark.gpu
def test_200_frame_window_feeds_grusage():
    from types import SimpleNamespace
    import sldm_gnn_b200 as sg
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    V, T, F = 120, 200, 6
    x = _traj(V, T, seed=21, spread=80.0, p_present=0.9).to(dev)
    ei, ea = sg.build_proximity_edges(x, 10.0)
    ei_r, ea_r = proximity_edges_oracle(x.cpu(), 10.0)
    assert ei.size(1) > V and torch.equal(ei.cpu(), ei_r) and torch.equal(ea.cpu(), ea_r)
    model = sg.GruSage(dynamic_features_num=F, frames_num=T, gru_hidden_size=32, gru_num_layers=1, fc1dims=[64],
                       sage_hidden_dims=[64, 64], fc2dims=[32], dropout=None, negative_slope=0.1,
                       map_included=False).to(dev)
    data = SimpleNamespace(x=x, xdims=torch.randn(V, 2, device=dev), xsttype=torch.randint(0, 9, (V,), device=dev),
                           pos_raw=x[:, :, :2].contiguous(), edge_index=ei,
                           batch=torch.zeros(V, dtype=torch.long, device=dev), num_graphs=1)
    out = model(data)
    assert out.shape == (1, 1) and bool(torch.isfinite(out).all())
    out.sum().backward()
    grads = [p.grad for p in model.parameters() if p.requires_grad]
    assert all(g is not None and bool(torch.isfinite(g).all()) for g in grads)
    assert all(float(p.grad.abs().sum()) > 0 for p in model.sage.parameters())
