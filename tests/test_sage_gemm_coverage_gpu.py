"""Every SageBlock GEMM kernel variant against fp64, at sizes where each persistent CTA runs several tiles.

The tensor-core kernels of sage_tc.cu are persistent: a CTA walks 128-row tiles (`tile += gridDim.x`) and carries its
rings across them -- the A and B operand rings, the TMEM A slots and accumulators, the drain -> finisher hand-off and,
in k_wgrad_tc, the accumulator flush groups -- each with its own mbarrier parity.  Which phase a chunk lands in depends
on the chunks per tile (2 Fin/32 forward, 2 Fout/32 DGRAD), so a parity slip shows only at some widths and only once a
CTA starts its second tile.  Each case (Fin, Fout) of CASES says which kernel instance it is there for;
expected_kernels() restates the eligibility rules, and every run asserts the launches with torch.profiler, so a case
cannot drift onto another path unnoticed.  Every case runs at three sizes (S = the device's SM count):

  N = 200                two tiles, one of them a tail
  N = 128 S + 1          one CTA runs a second tile: the one-row tail
  N = 5 * 128 S + 77     every CTA runs 5-6 forward tiles or 10-12 DGRAD work items, k_wgrad_tc >= 6 flush groups per
                         CTA, and the SIMT forward takes its large-N tile configuration

Each kernel is checked on its own inputs, so that a failure names the kernel and not the layer: the projection on
random agg / x; the LayerNorm/activation backward on the kernel's saved xhat / rstd; DGRAD and WGRAD on the kernel's own
dz.  The references are computed on the CPU in fp32 and fp64 (parity_util.assert_close: rtol 1e-5 / atol 1e-6, fp64
adjudication).  Checks that need no reference: the forward is bit-identical under a row permutation and for a prefix
of the rows, and every output and gradient is bit-identical whichever way the tensor kernels walk their tiles
(SLDM_TC_REVERSE).  The SIMT kernels (SLDM_DISABLE_TC=1, read once per process) run the same table in a subprocess:
`python tests/test_sage_gemm_coverage_gpu.py simt SIZE`; `... hashes` prints the digests of the tile-order check.
"""
import hashlib
import json
import math
import os
import re
import subprocess
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import sldm_gnn_b200 as sg  # noqa: E402
from sldm_gnn_b200 import ops  # noqa: E402
from parity_util import ATOL, assert_close  # noqa: E402

EPS, SLOPE = 1e-5, 0.1

# (Fin, Fout) -> what the case is there for.  NT = output column slabs of 32 (Fout forward, Fin DGRAD), Kc = 32-wide K
# chunks per source (Fin / 32 forward, Fout / 32 DGRAD), NB = column blocks of k_wgrad_tc (Fin / 32).
CASES = {
    (32, 16): "forward NT=1 with a partial slab, Kc=1",
    (32, 32): "forward NT=1, Kc=1; DGRAD NT=1 with the bulk store; MapEncoder width",
    (64, 48): "forward NT=2 with a partial slab, Kc=2",
    (96, 80): "forward NT=3 with a partial slab, Kc=3",
    (128, 96): "forward NT=3, Kc=4; DGRAD NT=4, Kc=3; GruSage's first block layer",
    (128, 112): "forward NT=4 with a partial slab, Kc=4",
    (128, 128): "forward NT=4, Kc=4; DGRAD NT=4, Kc=4; k_wgrad_tc<4>",
    (160, 64): "forward Kc=5 (backward on the SIMT kernels)",
    (256, 128): "forward Kc=8 (backward on the SIMT kernels)",
    (224, 16): "forward Kc=7, NT=1 (backward on the SIMT kernels)",
    (16, 32): "DGRAD NT=1, partial, st.global finisher; k_wgrad_tc<1> with a half block",
    (48, 64): "DGRAD NT=2, partial, st.global finisher",
    (80, 96): "DGRAD NT=3, partial, st.global finisher",
    (112, 128): "DGRAD NT=4, partial, st.global finisher",
    (48, 160): "DGRAD Kc=5 with k_ln_bwd_rows<2>",
    (128, 256): "DGRAD Kc=8 with k_ln_bwd_rows<2>",
    (20, 36): "k_wgrad_tc<1> with a partial block, M = 36",
    (36, 100): "k_wgrad_tc<2> with a partial block, M = 100",
    (68, 20): "k_wgrad_tc<3> with a partial block, M = 20",
    (124, 124): "k_wgrad_tc<4> with a partial block, M = 124",
    (13, 7): "SIMT only: odd widths",
    (200, 40): "SIMT only: Fin > 128",
    (8, 256): "SIMT only: Fout = 256",
    (96, 96): "GruSage's second block layer: forward NT=3, DGRAD NT=3, k_wgrad_tc<3>",
}
# bf16 feature storage (agg and x in bf16): k_sage_tc<NT, 0, true> for NT = 1..4, k_wgrad_tc<2 | 4, true>
BF16_CASES = ((64, 32), (64, 96), (128, 64), (128, 128))
SIZES = ("two_tiles", "one_cta_two_tiles", "many_tiles")


def sizes(sms: int) -> dict:
    return {"two_tiles": 200, "one_cta_two_tiles": 128 * sms + 1, "many_tiles": 5 * 128 * sms + 77}


def _slabs(F: int) -> int:
    return (F + 31) // 32


def expected_kernels(Fin: int, Fout: int, tc: bool = True, bf16: bool = False) -> set:
    """The GEMM and LayerNorm-backward kernels one project_forward + layer_backward(need_dx) launches: the eligibility
    rules of sage_tc.cu (project_forward_tc_eligible, dgrad_tc_eligible, wgrad_tc_eligible, their bf16 versions) and
    the dispatch of sage_bwd.cu, for 16-byte aligned buffers.  Names as routed_kernels() normalises them."""
    if bf16:
        return {f"k_sage_tc<{_slabs(Fout)},0,1>", "k_ln_bwd_rows<1>", f"k_sage_tc<{_slabs(Fin)},1,0>",
                f"k_wgrad_tc<{_slabs(Fin)},1>"}
    fwd = tc and Fin % 32 == 0 and Fin >= 32 and Fout % 16 == 0 and 16 <= Fout <= 128
    dgrad = tc and Fout % 32 == 0 and Fout >= 32 and Fin % 16 == 0 and 16 <= Fin <= 128
    wgrad = tc and Fin % 4 == 0 and Fout % 4 == 0 and 16 <= Fin <= 128 and 16 <= Fout <= 128
    ks = {f"k_sage_tc<{_slabs(Fout)},0,0>" if fwd else "k_sage_proj_fwd"}
    if dgrad:   # the LayerNorm backward streams on its own, the tensor kernel does both data-gradient GEMMs
        ks |= {f"k_ln_bwd_rows<{1 if Fout <= 128 else 2}>", f"k_sage_tc<{_slabs(Fin)},1,0>"}
    else:
        ks.add("k_ln_bwd_dgrad")
    ks.add(f"k_wgrad_tc<{_slabs(Fin)},0>" if wgrad else "k_wgrad")
    return ks


_ROUTED = ("k_sage_tc", "k_sage_proj_fwd", "k_ln_bwd_rows", "k_ln_bwd_dgrad", "k_wgrad_tc", "k_wgrad")
_SIMT_TILED = ("k_sage_proj_fwd", "k_ln_bwd_dgrad", "k_wgrad")   # template arguments are tile shapes: family only


def routed_kernels(names) -> set:
    """Kernel names from the profiler ('void sldm::k_sage_tc<3, 1, false>(...)') -> {'k_sage_tc<3,1,0>', ...}, only
    the kernels expected_kernels() speaks about; `false` / `0` and `true` / `1` are the same argument."""
    out = set()
    for n in names:
        m = re.search(r"(?<!\w)(k_\w+)(?:<([^<>]*)>)?", n)
        if not m or m.group(1) not in _ROUTED:
            continue
        fam, args = m.group(1), m.group(2)
        if fam in _SIMT_TILED or args is None:
            out.add(fam)
            continue
        norm = [{"false": "0", "true": "1"}.get(a.strip(), a.strip()) for a in args.split(",")]
        out.add(f"{fam}<{','.join(norm)}>")
    return out


# ------------------------------------------------------------------------------------------ CPU checks of the table --
def test_case_table_reaches_every_gemm_instance():
    reached = set().union(*(expected_kernels(*c) for c in CASES))
    reached |= set().union(*(expected_kernels(*c, bf16=True) for c in BF16_CASES))
    want = {f"k_sage_tc<{nt},{mode},0>" for nt in range(1, 5) for mode in (0, 1)}
    want |= {f"k_wgrad_tc<{nb},0>" for nb in range(1, 5)}
    want |= {f"k_sage_tc<{nt},0,1>" for nt in range(1, 5)} | {"k_wgrad_tc<2,1>", "k_wgrad_tc<4,1>"}
    assert want <= reached, sorted(want - reached)
    # the widths that leave the tensor path, and where they go
    assert expected_kernels(256, 128) == {"k_sage_tc<4,0,0>", "k_ln_bwd_dgrad", "k_wgrad"}
    assert expected_kernels(48, 160) == {"k_sage_proj_fwd", "k_ln_bwd_rows<2>", "k_sage_tc<2,1,0>", "k_wgrad"}
    assert expected_kernels(13, 7) == expected_kernels(200, 40) == expected_kernels(8, 256) == \
        {"k_sage_proj_fwd", "k_ln_bwd_dgrad", "k_wgrad"}
    for c in CASES:
        assert expected_kernels(*c, tc=False) == {"k_sage_proj_fwd", "k_ln_bwd_dgrad", "k_wgrad"}
    for Fin, Fout in BF16_CASES:      # the shapes the bf16 entry points take (sldm_sage_bf16_supported)
        assert Fin in (64, 128) and Fout % 32 == 0 and Fout <= 128
    assert routed_kernels(["void sldm::k_sage_tc<3, 1, false>(CUtensorMap_st, sldm::TcProblem)",
                           "sldm::k_wgrad_tc<2, true>(CUtensorMap_st)", "void sldm::k_wgrad(float const*)",
                           "void sldm::k_sage_proj_fwd<16, 8, 8>(float const*)", "void sldm::k_ln_bwd_rows<2>(float)",
                           "void sldm::k_split_weights(float const*)", "Memset (Device)"]) == \
        {"k_sage_tc<3,1,0>", "k_wgrad_tc<2,1>", "k_wgrad", "k_sage_proj_fwd", "k_ln_bwd_rows<2>"}


@pytest.mark.parametrize("sms", [148, 132, 160])
def test_sizes_put_several_tiles_on_every_cta(sms):
    """The three sizes do what they are chosen for (launch arithmetic of sage_tc.cu: one CTA per SM at most, 128-row
    tiles; k_wgrad_tc: 16-row chunks in whole flush groups of 8 per CTA)."""
    s = sizes(sms)
    tiles = {k: -(-n // 128) for k, n in s.items()}
    assert tiles["two_tiles"] == 2 and s["two_tiles"] % 128
    assert tiles["one_cta_two_tiles"] == sms + 1 and s["one_cta_two_tiles"] % 128 == 1
    t = tiles["many_tiles"]
    assert t // sms == 5 and -(-t // sms) == 6                      # forward: 5-6 tiles per CTA; DGRAD: 10-12 items
    chunks = -(-s["many_tiles"] // 16)                              # wgrad_tc_launch: 16-row chunks ...
    per_cta = -(-chunks // min(sms, chunks))
    cpc = -(-per_cta // 8) * 8                                      # ... in whole flush groups of 8 per CTA
    assert cpc // 8 >= 6                                            # every CTA but the last: >= 6 flush groups


# ------------------------------------------------------------------------------------------- inputs and references --
def make_case(Fin, Fout, N, bf16=False):
    """Parameters with the block's initialisation (U(+-1/sqrt(Fin))), LayerNorm affine gamma ~ U(0.5, 1.5) and
    beta ~ U(-0.5, 0.5), random agg / x / dout, a random graph with 5 edges per node (only its in-degrees matter)."""
    g = torch.Generator().manual_seed(7919 * Fin + 104729 * Fout + N + (1 if bf16 else 0))
    b = 1.0 / math.sqrt(Fin)

    def u(shape, lo, hi):
        return torch.rand(shape, generator=g) * (hi - lo) + lo
    p = dict(W_l=u((Fout, Fin), -b, b), b_l=u((Fout,), -b, b), W_r=u((Fout, Fin), -b, b),
             ln_w=u((Fout,), 0.5, 1.5), ln_b=u((Fout,), -0.5, 0.5))
    agg, x = torch.randn(N, Fin, generator=g), torch.randn(N, Fin, generator=g)
    if bf16:
        agg, x = agg.to(torch.bfloat16), x.to(torch.bfloat16)
    dout = torch.randn(N, Fout, generator=g)
    ei = torch.randint(0, N, (2, 5 * N), generator=g)
    return dict(p=p, agg=agg, x=x, dout=dout, ei=ei, N=N, Fin=Fin, Fout=Fout, bf16=bf16)


def forward_ref(c, dt):
    """z = agg W_l^T + b_l + x W_r^T, LayerNorm (biased variance), LeakyReLU -- from the (bf16-valued) inputs."""
    p = {k: v.to(dt) for k, v in c["p"].items()}
    z = c["agg"].to(dt) @ p["W_l"].T + p["b_l"] + c["x"].to(dt) @ p["W_r"].T
    mean = z.mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(((z - mean) ** 2).mean(1, keepdim=True) + EPS)
    xhat = (z - mean) * rstd
    y = xhat * p["ln_w"] + p["ln_b"]
    return dict(out=torch.where(y > 0, y, SLOPE * y), xhat=xhat, rstd=rstd[:, 0])


def ln_backward_ref(c, xhat, rstd, dt):
    """dz and the column sums from the kernel's own xhat / rstd.  The activation branch is taken on the sign of
    gamma * xhat + beta in fp64 (exact product, one rounding: the sign the kernels' fmaf sees) for both precisions."""
    p = c["p"]
    pos = xhat.double() * p["ln_w"].double() + p["ln_b"].double() > 0
    h, d, gam = xhat.to(dt), c["dout"].to(dt), p["ln_w"].to(dt)
    dy = torch.where(pos, d, d * SLOPE)
    t = dy * gam
    dz = rstd.to(dt)[:, None] * (t - t.mean(1, keepdim=True) - h * (t * h).mean(1, keepdim=True))
    return dict(dz=dz, db_l=dz.sum(0), dln_w=(dy * h).sum(0), dln_b=dy.sum(0))


def dgrad_ref(c, dz, dt):
    deg = torch.bincount(c["ei"][1], minlength=c["N"]).clamp(min=1).to(dt)
    dz = dz.to(dt)
    return dict(dagg=(dz @ c["p"]["W_l"].to(dt)) / deg[:, None], dxroot=dz @ c["p"]["W_r"].to(dt))


def wgrad_ref(c, dz, dt):
    dz = dz.to(dt)
    return dict(dW_l=dz.T @ c["agg"].to(dt), dW_r=dz.T @ c["x"].to(dt))


def bf16_ulp_distance(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """Distance in bf16 units of last place (monotone integer mapping of the bit patterns)."""
    def key(t):
        i = t.contiguous().view(torch.int16).to(torch.int32)
        return torch.where(i < 0, -(i & 0x7FFF), i)
    return (key(a) - key(b)).abs()


# ------------------------------------------------------------------------------------------------- running a case --
_RESULTS = ("out", "xhat", "rstd", "dz", "dagg", "dxroot", "dx", "dW_l", "db_l", "dW_r", "dln_w", "dln_b")


def run_kernels(c, dev, profile=True):
    """One project_forward and one layer_backward(need_dx) through ops, with the buffers kept so that dz, dagg and
    dxroot can be read back.  Returns (device tensors, the set of routed kernels launched | None)."""
    p = {k: v.to(dev) for k, v in c["p"].items()}
    agg, x, dout = c["agg"].to(dev), c["x"].to(dev), c["dout"].to(dev)
    csr = sg.build_csr(c["ei"].to(dev), c["N"])
    torch.cuda.synchronize()

    def launch():
        out, xhat, rstd = ops.project_forward(agg, x, p["W_l"], p["b_l"], p["W_r"], p["ln_w"], p["ln_b"], EPS, SLOPE,
                                              True)
        bufs = ops.backward_buffers(c["N"], c["Fin"], c["Fout"], csr.E, dev, need_dx=True)
        ops.layer_backward(dout, x, agg, xhat, rstd, csr, p["W_l"], p["W_r"], p["ln_w"], p["ln_b"], SLOPE, True,
                           bufs=bufs)
        torch.cuda.synchronize()
        return dict(out=out, xhat=xhat, rstd=rstd, **{k: bufs[k] for k in _RESULTS[3:]})

    if not profile:
        return dict(launch(), _agg=agg, _x=x, _p=p), None
    from torch.profiler import ProfilerActivity, profile as prof_ctx
    with prof_ctx(activities=[ProfilerActivity.CUDA]) as prof:
        res = launch()
    return dict(res, _agg=agg, _x=x, _p=p), routed_kernels(e.key for e in prof.key_averages())


def check_routing(launched, c, tc, what):
    """The launches the case is there for, and no others (SIMT: no k_sage_tc / k_wgrad_tc at all)."""
    want = expected_kernels(c["Fin"], c["Fout"], tc=tc, bf16=c["bf16"])
    assert launched == want, f"{what}: launched {sorted(launched)}, the case is there for {sorted(want)}"


def check_numerics(c, got, what):
    """Every kernel against the fp32 reference with fp64 adjudication, each on its own inputs."""
    g = {k: got[k].cpu() for k in _RESULTS}
    r32, r64 = forward_ref(c, torch.float32), forward_ref(c, torch.float64)
    if c["bf16"]:
        # out is rounded to bf16 once, from fp32: within one bf16 ulp of the exact value rounded -- or, next to 0,
        # where a bf16 ulp is finer than fp32 noise, within the project's atol of the exact value
        o64 = r64["out"]
        ulps = bf16_ulp_distance(g["out"], o64.to(torch.bfloat16))
        ok = (ulps <= 1) | ((g["out"].double() - o64).abs() <= ATOL)
        assert bool(ok.all()), (f"{what}: bf16 out {int((~ok).sum())} elements > 1 ulp from fp64, "
                                f"max {int(ulps.max())} ulp")
    else:
        assert_close(g["out"], r32["out"], f"{what} forward out", want64=r64["out"])
    assert_close(g["xhat"], r32["xhat"], f"{what} forward xhat", want64=r64["xhat"])
    assert_close(g["rstd"], r32["rstd"], f"{what} forward rstd", want64=r64["rstd"])

    l32, l64 = ln_backward_ref(c, g["xhat"], g["rstd"], torch.float32), ln_backward_ref(c, g["xhat"], g["rstd"], torch.float64)
    # rows with an element at the activation's kink would move by the slope factor if either side evaluated
    # gamma * xhat + beta with one more rounding: left out of the element-wise dz check (not of the sums)
    y = g["xhat"].double() * c["p"]["ln_w"].double() + c["p"]["ln_b"].double()
    rows = ~(y.abs() < 1e-6).any(1)
    assert_close(g["dz"][rows], l32["dz"][rows], f"{what} LN backward dz", want64=l64["dz"][rows])
    for k in ("db_l", "dln_w", "dln_b"):
        assert_close(g[k], l32[k], f"{what} LN backward {k}", scale_atol=True, want64=l64[k])

    d32, d64 = dgrad_ref(c, g["dz"], torch.float32), dgrad_ref(c, g["dz"], torch.float64)
    for k in ("dagg", "dxroot"):
        assert_close(g[k], d32[k], f"{what} DGRAD {k}", want64=d64[k])
    w32, w64 = wgrad_ref(c, g["dz"], torch.float32), wgrad_ref(c, g["dz"], torch.float64)
    for k in ("dW_l", "dW_r"):
        assert_close(g[k], w32[k], f"{what} WGRAD {k}", scale_atol=True, want64=w64[k])


def check_row_invariance(c, got, tc, what):
    """The forward of a row does not depend on where the row sits: bit-identical under a row permutation (every row
    moves to another tile, TMEM lane, slot and CTA) and, on the tensor path, for a prefix of the rows (another tile
    count, another tile -> CTA assignment)."""
    p, agg, x, N = got["_p"], got["_agg"], got["_x"], c["N"]

    def fwd(a, b):
        return ops.project_forward(a, b, p["W_l"], p["b_l"], p["W_r"], p["ln_w"], p["ln_b"], EPS, SLOPE, True)
    perm = torch.randperm(N, generator=torch.Generator().manual_seed(N)).to(agg.device)
    for name, a, b in zip(("out", "xhat", "rstd"), fwd(agg[perm], x[perm]), (got["out"], got["xhat"], got["rstd"])):
        assert torch.equal(a, b[perm]), f"{what}: forward {name} changes under a row permutation"
    if tc:
        n = N - N // 3
        for name, a, b in zip(("out", "xhat", "rstd"), fwd(agg[:n], x[:n]), (got["out"], got["xhat"], got["rstd"])):
            assert torch.equal(a, b[:n]), f"{what}: forward {name} of the first {n} rows differs from the full run"


def run_case(Fin, Fout, size, dev, tc, bf16=False):
    N = sizes(torch.cuda.get_device_properties(dev).multi_processor_count)[size]
    what = f"[{Fin}->{Fout}{' bf16' if bf16 else ''} N={N}{'' if tc else ' SIMT'}]"
    c = make_case(Fin, Fout, N, bf16=bf16)
    got, launched = run_kernels(c, dev)
    check_routing(launched, c, tc, what)
    check_row_invariance(c, got, tc, what)
    check_numerics(c, got, what)


# -------------------------------------------------------------------------------------------------------- GPU tests --
@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _case_id(c):
    return f"{c[0]}x{c[1]}"


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("case", list(CASES), ids=_case_id)
def test_tensor_path_kernels_match_fp64(dev, case, size):
    run_case(*case, size, dev, tc=True)


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("case", BF16_CASES, ids=_case_id)
def test_bf16_feature_kernels_match_fp64(dev, case, size):
    run_case(*case, size, dev, tc=True, bf16=True)


def _script(*args, env=None):
    r = subprocess.run([sys.executable, os.path.abspath(__file__), *args], env=dict(os.environ, **(env or {})),
                       capture_output=True, text=True, timeout=1800, cwd=ROOT)
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("size", SIZES)
def test_simt_path_kernels_match_fp64(size):
    """The same table on the FP32 SIMT kernels (SLDM_DISABLE_TC=1): no tensor kernel may launch."""
    r = _script("simt", size, env={"SLDM_DISABLE_TC": "1"})
    assert r.returncode == 0 and "SIMT_OK" in r.stdout, r.stdout[-6000:] + r.stderr[-4000:]


@pytest.mark.gpu
def test_tile_order_does_not_change_any_bit():
    """SLDM_TC_REVERSE (bit 0: forward, bit 1: DGRAD walk their tiles from the last to the first; default 1) at the
    largest size: every output and gradient is bit-identical in all walk orders."""
    res = {}
    for mask in (None, "0", "3"):
        r = _script("hashes", env={} if mask is None else {"SLDM_TC_REVERSE": mask})
        assert r.returncode == 0 and "HASHES" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
        res[mask] = json.loads(r.stdout.strip().splitlines()[-1].split(" ", 1)[1])
    assert len(res[None]) == len(CASES) + len(BF16_CASES)
    for mask in ("0", "3"):
        diff = {k: sorted(n for n in res[None][k] if res[None][k][n] != res[mask][k][n]) for k in res[None]}
        diff = {k: v for k, v in diff.items() if v}
        assert not diff, f"SLDM_TC_REVERSE={mask} changes {diff}"


class _Branch(torch.nn.Module):
    """LeakyReLU with its branch given: y where `pos`, slope * y elsewhere."""

    def __init__(self, slope, pos):
        super().__init__()
        self.slope, self.pos = slope, pos

    def forward(self, y):
        return torch.where(self.pos, y, self.slope * y)


@pytest.mark.gpu
@pytest.mark.parametrize("hdims", [[128, 96, 96], [32, 32, 32]], ids=["c2_block", "map_encoder"])
def test_block_at_model_size_matches_oracle(dev, hdims):
    """The whole block at the size the model runs it (1024 unit map graphs, ~205 k rows): GruSage's block
    SageBlock([128, 96, 96]) and the MapEncoder width, output, dx and every parameter gradient, on run_pair's inputs.

    With ~2e7 pre-activations per layer, a few lie within fp32 noise of zero.  There fp32 and fp64 can take different
    branches of the LeakyReLU, and the branch scales that element's gradient by 1 or by the slope.  The change spreads
    through its row's LayerNorm backward into dx: at [128, 96, 96] the fp32 oracle itself is 7e-2 away from fp64 there.
    That is no bar for the kernels, so both oracles take the branch the kernels took.  The test first asserts that
    the kernels' branch differs from fp64's only where |gamma * xhat + beta| is below fp32 noise."""
    from workloads import unit_map_graphs
    from oracle.sage_oracle import SageBlockOracle
    from test_gpu_parity import check_pair
    ei, _, N = unit_map_graphs(1024, seed=hdims[0] + hdims[1])
    assert N > 128 * 5 * torch.cuda.get_device_properties(dev).multi_processor_count
    # run_pair's construction, in its order (same parameters, inputs and upstream gradient)
    torch.manual_seed(0)
    ref = SageBlockOracle(hdims, negative_slope=SLOPE)
    with torch.no_grad():
        for post in ref.posts:
            post[0].weight.uniform_(0.5, 1.5)
            post[0].bias.uniform_(-0.5, 0.5)
    ref64 = SageBlockOracle(hdims, negative_slope=SLOPE).double()
    ref64.load_state_dict({k: v.double() for k, v in ref.state_dict().items()})
    ours = sg.SageBlock(hdims, negative_slope=SLOPE)
    ours.load_state_dict(ref.state_dict(), strict=True)
    ours.to(dev)
    x = torch.randn(N, hdims[0])

    # the branch every output element of the kernels took (the block's own per-layer calls)
    eid = ei.to(dev)
    csr = sg.build_csr(eid, N)
    h, pos = x.to(dev), []
    for conv, post in zip(ours.convs, ours.posts):
        _, h, _, _, _ = ops.layer_forward(h, csr, conv.lin_l.weight, conv.lin_l.bias, conv.lin_r.weight,
                                          post[0].weight, post[0].bias, post[0].eps, SLOPE, False)
        pos.append((h > 0).cpu())
    ys = []
    hooks = [post[0].register_forward_hook(lambda m, i, o: ys.append(o.detach())) for post in ref64.posts]
    with torch.no_grad():
        ref64(x.double(), ei)
    for hk in hooks:
        hk.remove()
    for l, (y, p) in enumerate(zip(ys, pos)):
        other = (y > 0) != p
        print(f"layer {l}: {int(other.sum())} of {y.numel()} branches differ from fp64, "
              f"max |y| there {float(y[other].abs().max()) if other.any() else 0.0:.2e}")
        assert bool((y[other].abs() < 1e-5).all()), f"layer {l}: the kernels' activation branch differs from fp64's " \
                                                    f"at |y| up to {float(y[other].abs().max()):.3e}"
    for blk in (ref, ref64):
        for post, p in zip(blk.posts, pos):
            post[1] = _Branch(SLOPE, p)

    xr = x.clone().requires_grad_(True)
    yr = ref(xr, ei)
    w = torch.randn_like(yr)
    (yr * w).sum().backward()
    xd = x.double().requires_grad_(True)
    yd = ref64(xd, ei)
    (yd * w.double()).sum().backward()
    xg = x.to(dev).requires_grad_(True)
    yg = ours(xg, eid)
    (yg * w.to(dev)).sum().backward()
    assert torch.equal(yg.detach(), h), "the block's output differs from its layer-by-layer forward"
    check_pair(ref, ours, (xr, yr), (xg, yg), ref64, (xd, yd))


# ----------------------------------------------------------------------------------------- subprocess entry point --
def _digests(got):
    return {k: hashlib.sha1(got[k].contiguous().view(torch.uint8).cpu().numpy().tobytes()).hexdigest() for k in _RESULTS}


def main(argv):
    dev = torch.device("cuda:0")
    if argv[0] == "simt":
        assert os.environ.get("SLDM_DISABLE_TC") == "1", "the SIMT run needs SLDM_DISABLE_TC=1"
        failures = []
        for Fin, Fout in CASES:
            try:
                run_case(Fin, Fout, argv[1], dev, tc=False)
            except AssertionError as e:
                failures.append(str(e))
        if failures:
            print("\n".join(failures))
            return 1
        print("SIMT_OK")
        return 0
    if argv[0] == "hashes":
        N = sizes(torch.cuda.get_device_properties(dev).multi_processor_count)["many_tiles"]
        out = {}
        for (Fin, Fout), bf16 in [(k, False) for k in CASES] + [(k, True) for k in BF16_CASES]:
            got, _ = run_kernels(make_case(Fin, Fout, N, bf16=bf16), dev, profile=False)
            out[f"{Fin}x{Fout}{' bf16' if bf16 else ''}"] = _digests(got)
        print("HASHES " + json.dumps(out))
        return 0
    raise SystemExit(f"usage: {sys.argv[0]} simt SIZE | hashes")


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
