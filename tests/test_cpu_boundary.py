"""CPU-side checks: the C-ABI library loads and exports every declared symbol, its parameter inventory
matches the reference's state_dict (via the golden key lists), host logic of the diffusion mirrors the oracle."""
import ctypes as C
import json
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from resshift_b200 import _lib
from resshift_b200.config import preset

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "resshift_b200.h").read_text()
    declared = set(re.findall(r"\b(rs_[a-z0-9_]+)\s*\(", header))
    declared -= {"rs_unet_config"}
    assert declared == set(_lib.declared_symbols())
    for name in declared:
        assert hasattr(_lib.lib, name), name
    assert _lib.lib.rs_version() >= 100


@pytest.mark.parametrize("name", ["realsr", "faceir", "inpaint"])
def test_engine_inventory_matches_reference_state_dict(golden_dir, name):
    gold = json.loads((golden_dir / f"unet_keys_{name}.json").read_text())
    ucfg, _ = preset(name)
    h = C.c_void_p()
    cfgc = _lib.make_config(ucfg)
    _lib.check(_lib.lib.rs_unet_create(C.byref(cfgc), C.byref(h)))
    try:
        n = _lib.lib.rs_unet_param_count(h)
        buf = C.create_string_buffer(256)
        shape = (C.c_int32 * 4)()
        nd, isb = C.c_int32(), C.c_int32()
        mine = []
        for i in range(n):
            _lib.check(_lib.lib.rs_unet_param_info(h, i, buf, 256, shape, C.byref(nd), C.byref(isb)))
            mine.append((buf.value.decode(), [shape[j] for j in range(nd.value)]))
        assert sorted(mine) == sorted((k, s) for k, s, _ in gold["entries"])
        assert _lib.lib.rs_unet_arena_bytes(h) > 2 * 0.95 * gold["n_params"]     # ~fp16 per parameter
    finally:
        _lib.lib.rs_unet_destroy(h)


def test_error_reporting_is_by_code_and_message():
    ucfg, _ = preset("tiny")
    cfgc = _lib.make_config(ucfg)
    cfgc.swin_heads = 5                      # head_dim != 32 -> rejected
    h = C.c_void_p()
    rc = _lib.lib.rs_unet_create(C.byref(cfgc), C.byref(h))
    assert rc < 0 and b"head_dim" in _lib.lib.rs_last_error()
    with pytest.raises(_lib.RsError):
        _lib.check(rc)


def test_module_state_dict_loads_reference_named_checkpoint(golden_dir):
    from resshift_b200.models.unet import UNetModelSwin
    from resshift_b200.weights import random_state_dict
    gold = json.loads((golden_dir / "unet_keys_realsr.json").read_text())
    ucfg, _ = preset("realsr")
    m = UNetModelSwin(**ucfg.to_kwargs())
    assert sorted(m.state_dict().keys()) == sorted(k for k, _, _ in gold["entries"])
    m.load_state_dict(random_state_dict(ucfg, 1), strict=True)
    # zero_module semantics of the reference constructor (models/unet.py:172-174) before loading
    m2 = UNetModelSwin(**ucfg.to_kwargs())
    assert float(m2.state_dict()["input_blocks.1.0.out_layers.3.weight"].abs().max()) == 0.0


def test_cpu_call_fails_loudly():
    from resshift_b200.models.unet import UNetModelSwin
    ucfg, _ = preset("tiny")
    m = UNetModelSwin(**ucfg.to_kwargs())
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 3, 64, 64), torch.zeros(1), lq=torch.zeros(1, 3, 64, 64))


def test_diffusion_tables_match_oracle():
    from oracle import diffusion_oracle as do
    from resshift_b200.models.script_util import create_gaussian_diffusion
    for name, steps in (("realsr", None), ("realsr_journal", None), ("realsr_journal", 15)):
        _, d = preset(name, steps)
        diff = create_gaussian_diffusion(**d.to_kwargs())
        tabs = do.schedule_tables(do.eta_schedule(d.steps, d.min_noise_level, d.etas_end, d.kappa, d.schedule_kwargs["power"]), d.kappa)
        np.testing.assert_allclose(diff.sqrt_etas, tabs["sqrt_etas"], rtol=1e-13)
        np.testing.assert_allclose(diff.posterior_mean_coef1, tabs["coef1"], rtol=1e-13)
        np.testing.assert_allclose(diff.posterior_mean_coef2, tabs["coef2"], rtol=1e-13)
        np.testing.assert_allclose(diff.posterior_log_variance_clipped, tabs["log_var"], rtol=1e-13)
        t = torch.arange(diff.num_timesteps)
        np.testing.assert_allclose(diff._scale_input(torch.ones(diff.num_timesteps, 1), t)[:, 0].numpy(), tabs["in_scale"], rtol=1e-6)


def test_timestep_respacing_map():
    from resshift_b200.models.script_util import create_gaussian_diffusion
    _, d = preset("realsr")
    d.timestep_respacing = 5
    diff = create_gaussian_diffusion(**d.to_kwargs())
    assert diff.num_timesteps == 5 and diff.timestep_map == [0, 3, 6, 9, 12]


def test_yaml_loader_resolves_interpolations(tmp_path):
    from resshift_b200.sampler import load_yaml
    p = tmp_path / "c.yaml"
    p.write_text("autoencoder:\n  params:\n    embed_dim: 3\nmodel:\n  params:\n    out_channels: ${autoencoder.params.embed_dim}\n    lq_size: 64\n")
    cfg = load_yaml(p)
    assert cfg.model.params.out_channels == 3 and cfg.model.params["lq_size"] == 64


def _tile_config(m_tiles, cout, num_kb):
    out = (C.c_int32 * 9)()
    _lib.check(_lib.lib.rs_debug_tile_config(m_tiles, cout, num_kb, out))
    keys = ("BN", "msub", "stages", "occ", "est_cycles", "cg", "splitk", "persist", "cluster_split")
    return dict(zip(keys, list(out)))


def test_tile_cost_model_invariants_for_the_model_layers():
    """Host-only: the conv launcher's cost model (launch.cuh) on the benchmark's layer shapes (batch 16).  Checks the
    structural rules the kernels rely on, not the timing estimates."""
    shapes = []           # (pixel tiles, Cout, k-blocks)
    for hw, cin, cout, k in [(64, 160, 160, 3), (64, 480, 160, 3), (64, 320, 320, 3), (64, 192, 576, 1), (64, 192, 192, 1),
                             (32, 320, 320, 3), (32, 640, 320, 3), (32, 192, 576, 1), (16, 320, 320, 3), (16, 960, 320, 3),
                             (16, 192, 576, 1), (8, 640, 640, 3), (8, 1280, 640, 3), (8, 192, 192, 1), (8, 640, 192, 1)]:
        shapes.append((16 * hw * hw // 128, cout, k * k * ((cin + 63) // 64)))
    for m_tiles, cout, nkb in shapes:
        tc = _tile_config(m_tiles, cout, nkb)
        cout16 = (cout + 15) // 16 * 16
        assert 16 <= tc["BN"] <= 256 and tc["BN"] % 16 == 0 and cout16 % tc["BN"] == 0, tc
        assert tc["cg"] in (1, 2) and tc["stages"] >= 2 and tc["splitk"] >= 1, tc
        if tc["persist"]:
            # only layers with at least two pixel tiles per SM (pair); double-buffered accumulators must fit in TMEM
            workers = 74 if tc["cg"] == 2 else 148
            assert (m_tiles + tc["cg"] - 1) // tc["cg"] >= 2 * workers and 2 * tc["BN"] <= 512 and tc["splitk"] == 1, tc
        if tc["cluster_split"]:
            assert tc["cg"] == 2 and tc["splitk"] == 2 and (tc["BN"] // 2) % 8 == 0 and not tc["persist"], tc
        if tc["splitk"] > 1:
            assert nkb // tc["splitk"] >= 6, tc            # every K range keeps a pipeline's worth of k-blocks
    # the 64x64 level runs persistent, the few-tile 3x3 layers split K
    assert _tile_config(512, 160, 27)["persist"] == 1
    assert _tile_config(8, 640, 90)["splitk"] > 1
    assert _tile_config(128, 320, 45)["persist"] == 0


def test_tile_starts_match_reference_image_splitter(golden_dir):
    """The sampler's tiling of large inputs must cut the same tiles as the reference's ImageSpliterTh
    (utils/util_image.py:889-979): the row / column starts it computed are stored in tests/golden/image_splitter.json
    (oracle/make_golden_splitter.py)."""
    from resshift_b200.sampler import tile_starts
    table = {(300, 128, 128): [0, 128, 172], (256, 128, 128): [0, 128], (240, 128, 112): [0, 112], (500, 128, 112): [0, 112, 224, 336, 372],
             (100, 128, 64): [0], (129, 128, 128): [0, 1], (592, 256, 224): [0, 224, 336], (448, 256, 224): [0, 192]}
    for (n, ps, st), want in table.items():
        assert tile_starts(n, ps, st) == want, (n, ps, st)
    cases = json.loads((golden_dir / "image_splitter.json").read_text())["tile_starts"]
    assert len(cases) == 82 * 6
    for c in cases:
        n, ps, st = c["n"], c["patch"], c["stride"]
        assert tile_starts(n, ps, st) == c["height_starts"], (n, ps, st)
        assert tile_starts(max(n // 2, 1), ps, st) == c["width_starts"], (n, ps, st)


def test_tile_plan_matches_reference_splitter(golden_dir):
    """Host side of the tiled pass: plan_tiles must enumerate exactly the tiles, in exactly the batches, that iterating
    the reference's ImageSpliterTh(extra_bs=chop_bs) yields (utils/util_image.py:889-960) — the per-call batch shape fixes
    the noise draw, the order fixes the overlap-average's summation order.  The reference's tiles are stored in
    tests/golden/image_splitter.json (oracle/make_golden_splitter.py).  (The device side — rs_op_tile_gather against
    the reference-form accumulate — is tests/test_gpu_vq.py::test_image_edges_match_torch and the tiled GPU test.)"""
    from resshift_b200.sampler import plan_tiles
    cases = json.loads((golden_dir / "image_splitter.json").read_text())["plan_tiles"]
    assert len(cases) == 6
    for c in cases:
        h, w, ps, st, bs = c["h"], c["w"], c["patch"], c["stride"], c["bs"]
        # (the reference's index_infos ends may exceed the image; its slice clips them)
        ref_groups = [[tuple(s) for s in grp] for grp in c["groups"]]
        ref_shapes = [tuple(s) for s in c["patch_shapes"]]
        hs_list, ws_list, th, tw, groups = plan_tiles(h, w, ps, st, bs)
        if h <= ps and w <= ps:                       # the reference does not tile at all in this case (sampler.py:186)
            assert groups == [[(0, 0)]]
            continue
        assert groups == ref_groups, (h, w, ps, st, bs)
        assert [(2 * len(g), th, tw) for g in groups] == ref_shapes, (h, w, ps, st, bs)
        assert hs_list == c["height_starts"] and ws_list == c["width_starts"]


def _stand_in_reference_tree(root: Path) -> Path:
    """A tree with the reference's layout where the overlay must take effect: top-level `sampler`, and a `models`
    namespace package (no __init__.py) holding `unet`, `script_util` and `basic_ops`.  The stand-ins define none of the
    names the probe reads, so a stand-in imported in place of the overlay fails the probe."""
    (root / "models").mkdir(parents=True)
    for rel in ("sampler.py", "models/unet.py", "models/script_util.py", "models/basic_ops.py"):
        (root / rel).write_text("FROM_REFERENCE_TREE = True\n")
    return root


def test_overlay_resolves_reference_module_names_to_this_package(tmp_path):
    """`python -m resshift_b200.launch <script>` must make `sampler`, `models.unet`, `models.script_util` resolve to this
    package while every other `models.*` module still comes from the reference tree (namespace package), exactly as an
    unmodified reference entry script imports them.  The reference tree is a stand-in with the same module layout."""
    import subprocess
    import sys
    ref_root = _stand_in_reference_tree(tmp_path / "reference")
    probe = tmp_path / "entry" / "probe_entry.py"
    probe.parent.mkdir()
    probe.write_text(
        "import sampler, models.unet, models.script_util\n"
        "import models.basic_ops as ref_ops\n"
        "print('sampler=' + sampler.ResShiftSampler.__module__)\n"
        "print('unet=' + models.unet.UNetModelSwin.__module__)\n"
        "print('diffusion=' + models.script_util.create_gaussian_diffusion.__module__)\n"
        "print('ref_ops=' + ref_ops.__file__)\n")
    # the probe sits in a scratch directory; the reference tree is appended the way its own scripts would see it
    env = dict(**__import__("os").environ, PYTHONPATH=str(ref_root) + ":" + str(ROOT / "oracle" / "_shims"))
    out = subprocess.run([sys.executable, "-m", "resshift_b200.launch", str(probe)], cwd=str(ROOT), env=env,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    got = dict(line.split("=", 1) for line in out.stdout.strip().splitlines() if "=" in line)
    assert got["sampler"] == "resshift_b200.sampler"
    assert got["unet"] == "resshift_b200.models.unet"
    assert got["diffusion"] == "resshift_b200.models.script_util"
    assert got["ref_ops"].startswith(str(ref_root))
