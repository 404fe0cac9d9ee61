"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every
symbol include/sldm_sage.h declares, the size/layout queries work without a GPU, the
module keeps the reference's constructor / state-dict contract, and the product path
refuses to run on the CPU (no fallback)."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest
import torch

import sldm_gnn_b200 as sg
from sldm_gnn_b200 import _lib
from oracle.sage_oracle import SageBlockOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "sldm_sage.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sldm_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    names = header_functions()
    assert len(names) >= 16
    lib = C.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/sldm_sage.h but not exported"
    assert sorted(_lib.EXPORTS) == names, "ctypes prototypes and header disagree"
    assert _lib.lib.sldm_abi_version() == 1


def test_library_is_sm100a_only_and_has_no_oracle_dependency():
    import subprocess
    out = subprocess.run(["cuobjdump", "--list-elf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs
    deps = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in deps and "torch" not in deps


def test_layout_and_workspace_queries_without_gpu():
    lay = _lib.csr_layout(1000, 5000)
    assert lay["meta"] == 0 and lay["total"] > 2 * 1001 + 2 * 5000
    offs = [lay[k] for k in _lib.CSR_SECTIONS]
    assert all(o % 64 == 0 for o in offs), "sections must be 256-byte aligned"
    assert lay["rowptr_src"] - lay["rowptr_dst"] >= 1001 and lay["col_dst"] - lay["col_src"] >= 5000
    assert _lib.lib.sldm_csr_workspace_bytes(1000, 5000) >= 6 * 5000 * 4
    assert _lib.lib.sldm_csr_workspace_bytes(-1, 0) == -1
    assert _lib.lib.sldm_segment_workspace_bytes(1000, 5000, 128) > 0
    assert _lib.lib.sldm_sage_layer_fwd_workspace_bytes(1000, 5000, 128, 96) >= 2 * 128 * 96 * 4
    assert _lib.lib.sldm_sage_layer_bwd_workspace_bytes(1000, 5000, 128, 96) >= 2 * 128 * 96 * 4
    with pytest.raises(ValueError):
        _lib.csr_layout(-1, 0)


def test_host_entry_fails_loudly_without_a_device():
    if torch.cuda.is_available():
        pytest.skip("has a GPU")
    x = np.zeros((4, 8), np.float32)
    ei = np.zeros((2, 3), np.int64)
    hd = (C.c_int32 * 2)(8, 8)
    bufs = [np.zeros(s, np.float32) for s in ((8, 8), (8,), (8, 8), (8,), (8,))]
    params = (C.c_void_p * 5)(*[b.ctypes.data for b in bufs])
    out = np.zeros((4, 8), np.float32)
    rc = _lib.lib.sldm_sage_block_forward_host(x.ctypes.data, ei.ctypes.data, 4, 3, hd, 1, params, 1e-5, 0.1, out.ctypes.data)
    assert rc == _lib.ENODEVICE
    with pytest.raises(RuntimeError, match="no CUDA device"):
        _lib.check(rc)


# --------------------------------------------------------------- module contract --
def test_state_dict_contract_matches_reference_fixture():
    g = torch.load(os.path.join(ROOT, "tests", "golden", "ref_vehicle_dims_relu.pt"))
    blk = sg.SageBlock(g["hdims"], dropout=None, negative_slope=g["slope"])
    assert list(blk.state_dict().keys()) == list(g["state_dict"].keys())
    for k, v in blk.state_dict().items():
        assert v.shape == g["state_dict"][k].shape and v.dtype == torch.float32, k
    blk.load_state_dict(g["state_dict"], strict=True)
    # and back into the oracle, strictly (SURVEY 8c v)
    SageBlockOracle(g["hdims"]).load_state_dict(blk.state_dict(), strict=True)
    assert "convs.0.lin_r.bias" not in blk.state_dict()


def test_constructor_contract():
    with pytest.raises(AssertionError):
        sg.SageBlock([])
    blk = sg.SageBlock([128, 96, 96], dropout=0.25, negative_slope=0.1)
    assert len(blk.convs) == 2 and len(blk.posts) == 2
    assert isinstance(blk.posts[0][0], torch.nn.LayerNorm) and blk.posts[0][0].normalized_shape == (96,)
    assert isinstance(blk.posts[0][1], torch.nn.LeakyReLU) and blk.posts[0][1].negative_slope == 0.1
    assert isinstance(blk.posts[0][2], torch.nn.Dropout) and blk.posts[0][2].p == 0.25
    assert isinstance(sg.SageBlock([4, 4]).posts[0][1], torch.nn.ReLU)
    assert isinstance(sg.SageBlock([4, 4]).posts[0][2], torch.nn.Identity)
    n_params = sum(p.numel() for p in blk.parameters())
    assert n_params == 43584  # SURVEY 8a a1: [128,96,96]
    w = blk.convs[0].lin_l.weight
    assert w.abs().max() <= 1 / np.sqrt(128) + 1e-7


def test_identity_block_and_no_cpu_fallback():
    x = torch.randn(5, 3)
    ei = torch.randint(0, 5, (2, 7))
    assert sg.SageBlock([3])(x, ei) is x          # zero layers: identity, like the reference
    blk = sg.SageBlock([3, 4])
    with pytest.raises(RuntimeError, match="CUDA only"):
        blk(x, ei)
    with pytest.raises(RuntimeError, match="CUDA only"):
        sg.build_csr(ei, 5)


def test_edge_index_validation_matches_pyg():
    blk = sg.SageBlock([3, 4])
    x = torch.randn(5, 3)
    for bad in (torch.zeros((2, 3), dtype=torch.int32), torch.zeros((3,), dtype=torch.long),
                torch.zeros((3, 3), dtype=torch.long), [[0, 1], [1, 0]]):
        with pytest.raises(ValueError):
            blk(x, bad)


def test_forward_accepts_optional_batch_argument():
    import inspect
    sig = inspect.signature(sg.SageBlock.forward)
    assert list(sig.parameters)[:3] == ["self", "x", "edge_index"]
    assert sig.parameters["batch"].default is None


def test_reference_import_path_shim():
    mod = sg.install_reference_shim()
    assert sys.modules["src.models.blocks.sageblock"] is mod
    from importlib import import_module
    assert import_module("src.models.blocks.sageblock").SageBlock is sg.SageBlock
    del sys.modules["src.models.blocks.sageblock"]


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "sldm_gnn_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("no CPU", ""), f"{f} mentions the oracle"


def test_extras_shim_registers_the_reference_model_imports():
    """install_reference_shim(extras=True) puts our SageBlock, MapSpatialAttention and graph pools under the module names
    the reference's src/models/grusage.py imports them from (the pools only when torch_geometric itself is absent), so
    that file builds its GruSage from our components.  The parameter layout of that GruSage is checked against the
    reference's stored state dicts in tests/test_grusage.py."""
    import importlib
    owned = lambda k: k.split(".")[0] in ("src", "torch_geometric")
    saved = {k: v for k, v in sys.modules.items() if owned(k)}
    for k in saved:
        del sys.modules[k]
    try:
        try:
            import torch_geometric  # noqa: F401
            have_pyg = True
        except ImportError:
            have_pyg = False
        sg.install_reference_shim(extras=True)
        assert importlib.import_module("src.models.blocks.sageblock").SageBlock is sg.SageBlock
        assert importlib.import_module("src.models.map.mapattention").MapSpatialAttention is sg.MapSpatialAttention
        pools = importlib.import_module("torch_geometric.nn")
        if not have_pyg:
            assert pools.global_mean_pool is sg.global_mean_pool and pools.global_max_pool is sg.global_max_pool
    finally:
        for k in [k for k in sys.modules if owned(k)]:
            del sys.modules[k]
        sys.modules.update(saved)
