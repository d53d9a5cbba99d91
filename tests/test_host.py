"""CPU: host-side logic and the C-ABI surface (no GPU compute)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from dmnerf_b200 import synth, _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_abi_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "dmnerf_b200.h")).read()
    declared = set(re.findall(r"DMNERF_API[^;(]*?\b(dmnerf_\w+)\s*\(", hdr))
    assert len(declared) >= 14
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.dmnerf_abi_version() == 1
    assert ctypes.sizeof(_lib.RenderIO) == 20 * 8


def test_calls_fail_loudly_without_gpu(lib):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    h = ctypes.c_void_p()
    rc = lib.dmnerf_ctx_create(0, ctypes.byref(h))
    assert rc != 0 and len(lib.dmnerf_last_error()) > 0
    from dmnerf_b200.engine import get_context
    with pytest.raises(RuntimeError):
        get_context("cpu")
    from dmnerf_b200.embedder import get_embedder
    with pytest.raises(RuntimeError):
        get_embedder(10)[0].embed(torch.zeros(4, 3))


def test_layer_table_matches_reference_counts():
    assert synth.macs_per_sample(13) == 693504                     # SURVEY.md 8d
    assert abs(synth.flops_per_ray(13) - 355.07e6) < 0.01e6
    assert abs(synth.flops_per_ray(59) - 358.09e6) < 0.01e6
    w = synth.make_weights(3, 13)
    assert sum(v.size for v in w.values()) == 696338
    assert list(w) == synth.param_names(13) and len(w) == _lib.N_PARAMS
    assert synth.algorithmic_bytes_per_ray(13) == 96 and synth.algorithmic_bytes_per_ray(59) == 280


def test_model_has_reference_state_dict_layout():
    from dmnerf_b200.model import DM_NeRF
    m = DM_NeRF(8, 256, 63, 27, [4], 13)
    sd = m.state_dict()
    assert list(sd) == synth.param_names(13)
    assert tuple(sd["mlps.5.weight"].shape) == (256, 319) and tuple(sd["rgb_feature_linears.0.weight"].shape) == (128, 283)
    assert tuple(sd["ins_linear.weight"].shape) == (14, 128)
    with pytest.raises(NotImplementedError):
        DM_NeRF(4, 128, 63, 27, [2], 13)


def test_linspace_formula_used_by_the_kernel_matches_torch():
    # ray_ops.cuh: linspace01(i, n) -- emulate in float32
    for n in (128, 64, 5, 192):
        step = np.float32(1.0) / np.float32(n - 1)
        mine = np.array([step * np.float32(i) if i < n // 2 else np.float32(1.0 - np.float64(step) * (n - 1 - i))   # fma
                         for i in range(n)], dtype=np.float32)
        np.testing.assert_array_equal(mine, torch.linspace(0.0, 1.0, n).numpy())


def test_dropin_networks_package_exposes_reference_names():
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "dm-nerf_b200", "dropin"), ROOT]))
    code = ("from networks.render import dm_nerf, render_train;"
            "from networks.dm_nerf import get_embedder, DM_NeRF, Embedder;"
            "from networks.helpers import get_rays_k, z_val_sample, sample_pdf;"
            "from networks.penalizer import ins_penalizer, emptiness_penalizer;"
            "from networks.manipulator import exchanger, manipulator_render, manipulator_nerf, manipulator;"
            "from networks.helpers import get_select_full, get_select_crop;"
            "from networks.evaluator import ins_criterion, img2mse, mse2psnr, to8b, hungarian;"
            "e, d = get_embedder(10); assert d == 63; assert get_embedder(4)[1] == 27;"
            "import torch.nn as nn; assert isinstance(get_embedder(0, -1)[0], nn.Identity);"
            "print('ok')")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd="/tmp")
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr


# A stand-in for a DM-NeRF checkout's networks/ package: the module and function names the drop-in resolves, each function
# returning the callees it finds through its own module globals, and the same cross-module import lines as the original
# (manipulator and tester import from networks.helpers / networks.evaluator / networks.render).
STAND_IN_NETWORKS = {
    "helpers.py": """
def get_rays_k(H, W, K, c2w): return "stand-in"
def get_select_full(*args): return get_rays_k
def get_select_crop(*args): return get_rays_k
def z_val_sample(*args): return "stand-in"
def sample_pdf(*args): return "stand-in"
def get_rays(*args): return get_rays_k, sample_pdf
""",
    "evaluator.py": """
def hungarian(*args): return "stand-in"
def ins_criterion(*args): return hungarian
def to8b(x): return x
def calculate_ap(*args): return "stand-in"
def ins_eval(*args): return hungarian
""",
    "manipulator.py": """
from networks.evaluator import to8b, ins_eval
from networks.helpers import get_rays_k, sample_pdf
def exchanger(*args): return "stand-in"
def manipulator_render(*args): return "stand-in"
def manipulator_nerf(*args): return "stand-in"
def manipulator(*args): return manipulator_nerf, manipulator_render, exchanger
def manipulator_eval(*args): return manipulator, exchanger, get_rays_k, sample_pdf
def manipulator_demo(*args): return manipulator, exchanger, get_rays_k, sample_pdf
""",
    "tester.py": """
from networks.render import dm_nerf
from networks.evaluator import to8b, ins_eval
from networks.helpers import get_rays_k, z_val_sample
def render_test(*args): return dm_nerf, get_rays_k, z_val_sample
""",
}


def test_dropin_rebinds_native_functions_inside_the_reference_modules(tmp_path):
    """The reference drivers (manipulator_eval / manipulator_demo, get_select_*; train_*.py through networks.evaluator)
    resolve their callees through their OWN module globals: the drop-in must rebind the native functions there, not only
    re-export them.  DMNERF_REFERENCE_ROOT points at a stand-in checkout with the reference's module layout."""
    ref = tmp_path / "reference"
    (ref / "networks").mkdir(parents=True)
    for name, src in STAND_IN_NETWORKS.items():
        (ref / "networks" / name).write_text(src)
    env = dict(os.environ, DMNERF_REFERENCE_ROOT=str(ref),
               PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "dm-nerf_b200", "dropin"), ROOT]))
    code = r"""
import dmnerf_b200.manipulator as nm, dmnerf_b200.helpers as nh, dmnerf_b200.evaluator as ne, dmnerf_b200.render as nr
import networks.manipulator as M, networks.helpers as H, networks.evaluator as E
assert M.manipulator is nm.manipulator and M.exchanger is nm.exchanger
for fn in (M.manipulator_eval, M.manipulator_demo):
    g = fn.__globals__
    assert g["manipulator"] is nm.manipulator and g["exchanger"] is nm.exchanger, fn
    assert g["get_rays_k"] is nh.get_rays_k and g["sample_pdf"] is nh.sample_pdf, fn
    assert fn() == (nm.manipulator, nm.exchanger, nh.get_rays_k, nh.sample_pdf), fn
assert H.get_select_full is nh.get_select_full and H.get_select_crop is nh.get_select_crop and H.get_rays_k is nh.get_rays_k
assert H.get_rays() == (nh.get_rays_k, nh.sample_pdf)      # a reference helper the drop-in keeps calls the native callees
assert E.ins_criterion is ne.ins_criterion and callable(E.ins_eval) and callable(E.calculate_ap)
import networks.tester as T                       # the reference's test loop, resolved through the package __path__
assert T.dm_nerf is nr.dm_nerf and T.get_rays_k is nh.get_rays_k and T.z_val_sample is nh.z_val_sample
assert T.render_test() == (nr.dm_nerf, nh.get_rays_k, nh.z_val_sample)
print("ok")
"""
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-3000:]


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "dm-nerf_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), os.path.join(dp, f)


def test_z_val_sample_matches_reference_formula(golden_dir):
    from dmnerf_b200.helpers import z_val_sample
    g = dict(np.load(os.path.join(golden_dir, "rays.npz")))
    z = z_val_sample(7, 4.0, 15.0, 64)
    assert z.shape == (7, 64) and z.stride(0) == 0
    np.testing.assert_array_equal(z[3].numpy(), g["z"])
    np.testing.assert_array_equal(z_val_sample(2, 0.0, 6.5, 64)[1].numpy(), g["z_replica"])


def test_lazy_render_dict_behaves_like_a_dict():
    """dm_nerf()'s inference result: the lazily produced per-sample tensors must show up through every dict access path."""
    from dmnerf_b200.render import LazyRenderDict
    calls = []

    def rerender():
        calls.append(1)
        return {"rgb_fine": "again", "raw_fine": "RF", "raw_coarse": "RC", "z_vals_fine": "ZF", "z_vals_coarse": "ZC",
                "weights_fine": "WF", "weights_coarse": "WC"}

    d = LazyRenderDict({"rgb_fine": "fused", "depth_fine": "D"}, rerender)
    assert "raw_fine" in d and not calls                     # membership does not trigger the second render
    assert d["rgb_fine"] == "fused" and not calls
    assert d.get("raw_fine") == "RF" and calls == [1]
    assert d["rgb_fine"] == "fused"                          # existing entries are kept
    assert set(d) >= {"raw_coarse", "z_vals_fine", "weights_coarse", "rgb_fine"} and len(d) == 8 and calls == [1]
    d2 = LazyRenderDict({"rgb_fine": "fused"}, rerender)
    assert "RF" in list(d2.values()) and d2.get("nope", 7) == 7
    with pytest.raises(KeyError):
        d2["nope"]


def test_hungarian_host_logic_matches_the_oracle():
    """The host half of the matched instance loss (assignment on the valid rows + unmatched channels appended, evaluator.py:42-50)
    and the dense-gt -> row-index conversion, against the oracle's restatement on random cost matrices."""
    from dmnerf_b200.evaluator import _reorder, _rows_of_dense_gt
    from oracle import dmnerf_oracle as O
    gen = torch.Generator().manual_seed(4)
    for k, valid in ((13, 6), (59, 20), (6, 6)):
        cost = torch.rand(k, k, generator=gen)
        rows, cols = _reorder(cost, valid, k)
        from scipy.optimize import linear_sum_assignment
        r2, c2 = linear_sum_assignment(cost[:valid].numpy())
        assert list(rows) == list(r2) and list(cols[:valid]) == list(c2)
        assert sorted(cols) == list(range(k))
    lab = torch.tensor([3, 0, 3, 7, 0])
    valid = torch.unique(lab)
    gt = torch.zeros(5, 9)
    gt[:, :3] = torch.nn.functional.one_hot(lab)[..., valid].float()
    assert _rows_of_dense_gt(gt).tolist() == [1, 0, 1, 2, 0]
    gt[4] = 0
    assert _rows_of_dense_gt(gt).tolist() == [1, 0, 1, 2, -1]
    # and the oracle's ins_criterion runs on the same tiny case (sanity of the fixture generator's path)
    pred = torch.sigmoid(torch.randn(5, 9, generator=gen))
    assert np.isfinite(float(O.ins_criterion(pred, lab.float(), 9)[0].sum()))


def test_shipped_library_hot_kernels_are_tcgen05_code():
    """cuobjdump -sass of the built library (no GPU needed): the network, gradient-chain and weight-gradient kernels issue
    tcgen05.mma (UTCHMMA) with tensor-memory loads (LDTM); the persistent kernels stream their weights with the bulk-copy engine
    (UBLKCP); no legacy mma.sync (HMMA) anywhere.  The counts are committed in profiles/r02_sass_histogram.txt."""
    import re
    import shutil
    import subprocess
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    path = os.path.join(ROOT, "dm-nerf_b200", "lib", "libdmnerf_b200.so")
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    per, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = per.setdefault(m.group(1), {"UTCHMMA": 0, "LDTM": 0, "STTM": 0, "UBLKCP": 0, "HMMA": 0})
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur is not None and m.group(1) in cur:
            cur[m.group(1)] += 1
    assert per, "no kernels found in the library"
    assert sum(c["HMMA"] for c in per.values()) == 0
    hot = {"mlp_umma_kernel": 2, "bwd_chain_kernel": 1, "gemm_tn_tc_kernel": 4, "gemm_nn_tc_kernel": 3}
    for name, n_inst in hot.items():
        ks = [c for k, c in per.items() if name in k]
        assert len(ks) == n_inst, (name, len(ks))
        for c in ks:
            assert c["UTCHMMA"] > 0 and c["LDTM"] > 0, (name, c)
    for name in ("mlp_umma_kernel", "bwd_chain_kernel"):
        for k, c in per.items():
            if name in k:
                assert c["UBLKCP"] > 0 and c["STTM"] > 0, (name, c)


def test_integration_doc_names_every_exported_symbol():
    """INTEGRATION.md section 1 maps every entry point of include/dmnerf_b200.h to the reference interface it replaces."""
    header = open(os.path.join(ROOT, "include", "dmnerf_b200.h")).read()
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    syms = sorted(set(re.findall(r"DMNERF_API\s+[\w\s\*]+?\b(dmnerf_\w+)\s*\(", header)))
    assert len(syms) >= 40
    missing = [s for s in syms if s not in doc]
    assert not missing, missing
