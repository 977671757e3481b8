"""CPU: host-side mirror of the reference interface, the C-ABI surface, synthetic data, sharding."""
import ctypes
import os
import re
import sys
import types

import numpy as np
import pytest
import torch

from conftest import DEFAULT_ARGS, VARIANT_ARGS, ROOT
import drawingspinup_b200 as dsu
from drawingspinup_b200 import capi, synth
from drawingspinup_b200.pipeline import shard_range
from oracle import reference_port as rp


# ---------------------------------------------------------------- state-dict contract (SURVEY 8a row a8)
@pytest.mark.parametrize("stage,cls", [(1, dsu.GeneratorJ_RIC), (2, dsu.GeneratorJ)])
def test_state_dict_layout_matches_reference(stage, cls):
    m = cls(**DEFAULT_ARGS)
    sd = m.state_dict()
    ref = synth.make_state_dict(stage)
    assert len(sd) == 89
    assert list(sd.keys()) == list(ref.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(ref[k].shape), k
    k0 = 3 if stage == 1 else 7
    assert tuple(sd["conv0.conv.weight"].shape) == (32, 6, k0, k0)
    assert tuple(sd["conv_11.0.weight"].shape) == (64, 166, k0, k0)
    assert sd["conv0.normalization.num_batches_tracked"].dtype == torch.int64
    assert sum(v.numel() for k, v in sd.items() if v.dtype != torch.int64 and "running" not in k) == \
        (3279427 if stage == 2 else 3279427 - 32 * 6 * 40 - 64 * 166 * 40)


@pytest.mark.parametrize("cls", [dsu.GeneratorJ_RIC, dsu.GeneratorJ])
def test_strict_load_and_round_trip(cls):
    stage = 1 if cls is dsu.GeneratorJ_RIC else 2
    m = cls(**DEFAULT_ARGS)
    sd = synth.to_torch_state_dict(synth.make_state_dict(stage, seed=5))
    m.load_state_dict(sd)                               # strict=True
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k]), k
    bad = dict(sd)
    bad.pop("conv_12.0.bias")
    with pytest.raises(RuntimeError):
        m.load_state_dict(bad)
    bad = dict(sd)
    bad["extra.weight"] = torch.zeros(1)
    with pytest.raises(RuntimeError):
        m.load_state_dict(bad)


def test_reference_constructor_signature_and_defaults():
    import inspect
    sig = inspect.signature(dsu.GeneratorJ.__init__)
    names = list(sig.parameters)[1:9]
    assert names == ["norm_layer", "gpu_ids", "use_bias", "resnet_blocks", "tanh", "filters", "input_channels", "append_smoothers"]
    d = {k: sig.parameters[k].default for k in names}
    assert d == dict(norm_layer="batch_norm", gpu_ids=None, use_bias=False, resnet_blocks=9, tanh=False,
                     filters=(64, 128, 128, 128, 128, 64), input_channels=3, append_smoothers=False)
    m = dsu.GeneratorJ()                                # reference defaults: 9 blocks, no tanh, no smoothers
    assert "conv_12.weight" in m.state_dict() and "conv_11_a.0.weight" not in m.state_dict()
    assert len([k for k in m.state_dict() if k.startswith("resnets.8.")]) > 0


def test_variant_config_keys():
    m = dsu.GeneratorJ(**VARIANT_ARGS)
    keys = list(m.state_dict().keys())
    ref = list(synth.make_state_dict(2, filters=VARIANT_ARGS["filters"], resnet_blocks=2, input_channels=5, tanh=False,
                                     append_smoothers=False, use_bias=True).keys())
    assert keys == ref


def test_unsupported_options_fail_loudly():
    m = dsu.GeneratorJ(norm_layer="instance_norm", **DEFAULT_ARGS)         # nn.InstanceNorm2d has no state: only conv_11_a.2 remains
    keys = list(m.state_dict().keys())
    assert keys == list(synth.make_state_dict(2, norm="instance_norm").keys()) and len(keys) == 29
    assert list(dsu.GeneratorJ_RIC(norm_layer=None, **DEFAULT_ARGS).state_dict().keys()) == list(synth.make_state_dict(1, norm="none").keys())
    with torch.no_grad(), pytest.raises(IndexError):                          # the reference's own stage-1 forward fails the same way
        dsu.GeneratorJ_RIC(norm_layer=None, **DEFAULT_ARGS).eval()(torch.zeros(1, 6, 16, 16))
    with pytest.raises(AssertionError):
        dsu.GeneratorJ(norm_layer="layer_norm")
    with pytest.raises(ValueError):
        dsu.GeneratorJ(precision="fp8")


def test_no_cpu_fallback():
    m = dsu.GeneratorJ(**DEFAULT_ARGS).eval()
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 6, 16, 16))
    m.train()
    with pytest.raises(RuntimeError, match="inference-only"):
        m(torch.zeros(1, 6, 16, 16))


def test_install_rebinds_reference_names():
    fake = types.ModuleType("training.models")
    fake.GeneratorJ = object
    fake.GeneratorJ_RIC = object
    dsu.install(fake)
    assert fake.GeneratorJ is dsu.GeneratorJ and fake.GeneratorJ_RIC is dsu.GeneratorJ_RIC
    # build_model's lookup (trainers.py:33-35): getattr(m, model_type)(**args)
    model = getattr(fake, "GeneratorJ_RIC")(**DEFAULT_ARGS)
    assert isinstance(model, dsu.GeneratorJ_RIC)


def test_factory_seam_builds_engine_classes_with_reference_state_dict_layout(golden_dir):
    """The factory seam (trainers.py:33-35, ``getattr(training.models, name)(**args).to(device)``): after install() it
    constructs the engine classes, whose state dicts have exactly the layout of the models the reference's own
    build_model makes (89 keys in the same order, same shapes and dtypes; recorded by oracle/make_golden.py) and load
    such a state dict strictly; uninstall() restores the module's own classes."""
    import json
    from collections import OrderedDict
    with open(os.path.join(golden_dir, "reference_state_dict_layout.json")) as f:
        g = json.load(f)
    assert g["args"] == DEFAULT_ARGS
    originals = {name: type(name, (), {}) for name in ("GeneratorJ", "GeneratorJ_RIC")}
    m = types.ModuleType("training.models")
    m.__dict__.update(originals)
    dsu.install(m)
    gen = torch.Generator().manual_seed(0)
    for name, cls in (("GeneratorJ", dsu.GeneratorJ), ("GeneratorJ_RIC", dsu.GeneratorJ_RIC)):
        eng = getattr(m, name)(**dict(g["args"])).to("cpu")
        assert type(eng) is cls
        layout = g["models"][name]
        assert len(layout) == 89
        assert [[k, list(v.shape), str(v.dtype)] for k, v in eng.state_dict().items()] == layout
        sd = OrderedDict((k, torch.randint(0, 100, s, generator=gen) if dt == "torch.int64" else torch.randn(s, generator=gen))
                         for k, s, dt in layout)
        eng.load_state_dict(sd)                                       # strict
        assert all(torch.equal(a, b) for a, b in zip(eng.state_dict().values(), sd.values()))
    dsu.uninstall(m)
    assert all(getattr(m, name) is cls for name, cls in originals.items())


def test_launcher_runs_script_with_rebound_classes(tmp_path, monkeypatch, capsys):
    """drawingspinup_b200.run on a miniature stand-in for 3_style_translator: the script resolves the
    class through training.models exactly like trainers.build_model does."""
    pkg = tmp_path / "training"
    pkg.mkdir()
    (pkg / "models.py").write_text("class GeneratorJ: pass\nclass GeneratorJ_RIC: pass\n")
    (tmp_path / "script.py").write_text(
        "import sys, training.models as m\n"
        "g = getattr(m, 'GeneratorJ')(input_channels=6)\n"
        "print('CLASS', type(g).__module__, len(g.state_dict()), sys.argv[1:])\n")
    from drawingspinup_b200 import run
    monkeypatch.setattr(sys, "argv", list(sys.argv))
    cwd = os.getcwd()
    for k in [k for k in sys.modules if k == "training" or k.startswith("training.")]:
        monkeypatch.delitem(sys.modules, k)
    try:
        assert run.main([str(tmp_path / "script.py"), "--uid", "abc"]) == 0
    finally:
        os.chdir(cwd)
        for k in [k for k in sys.modules if k == "training" or k.startswith("training.")]:
            sys.modules.pop(k)
        if str(tmp_path) in sys.path:
            sys.path.remove(str(tmp_path))
    out = capsys.readouterr().out
    assert "CLASS drawingspinup_b200.models" in out and "['--uid', 'abc']" in out


# ---------------------------------------------------------------- RIC offsets: product restatement == oracle == golden
def test_package_ric_offsets_bit_identical_to_oracle(golden_dir):
    for h, w in ((24, 20), (16, 16), (33, 12)):
        assert torch.equal(dsu.ric_offsets(h, w), rp.ric_offsets(h, w))
    g = np.load(os.path.join(golden_dir, "ric_coords_24x20.npz"))
    assert np.array_equal(dsu.ric_offsets(24, 20).numpy(), g["coords"])


# ---------------------------------------------------------------- C ABI surface
def _header_functions():
    text = open(os.path.join(ROOT, "include", "dsu_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dsu_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(built_lib):
    lib = ctypes.CDLL(built_lib)
    names = _header_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), "missing export " + n
    assert sorted(capi.SYMBOLS) == names                # the ctypes table covers the whole header
    assert b"sm_100a" in capi.lib().dsu_version()


def test_c_abi_rejects_bad_arguments_without_gpu(built_lib):
    lib = capi.lib()
    h = ctypes.c_void_p()
    assert lib.dsu_create(None, ctypes.byref(h)) < 0 and "null" in capi.last_error()
    cfg = capi.DsuConfig()
    cfg.kind = 7
    assert lib.dsu_create(ctypes.byref(cfg), ctypes.byref(h)) == -1
    cfg.kind = capi.KIND_GENERATORJ
    cfg.norm = 3                                        # DSU_NORM_NONE / BATCH / INSTANCE are 0 / 1 / 2
    assert lib.dsu_create(ctypes.byref(cfg), ctypes.byref(h)) == -1 and "norm" in capi.last_error()
    assert lib.dsu_forward(None, None, 1, 16, 16, None, None) < 0
    assert lib.dsu_to_image_space(None, None, 4, None) < 0
    lib.dsu_destroy(None)                               # no-op, must not crash


def test_missing_library_message(monkeypatch):
    monkeypatch.setattr(capi, "_lib", None)
    monkeypatch.setattr(capi, "LIB_PATH", "/nonexistent/libdsu_b200.so")
    with pytest.raises(RuntimeError, match="no CPU or PyTorch fallback"):
        capi.lib()


# ---------------------------------------------------------------- frame sharding (SURVEY 8e)
@pytest.mark.parametrize("n,world", [(64, 1), (64, 8), (339, 8), (210, 4), (5, 8), (0, 2), (256, 2)])
def test_shard_ranges_tile_the_sequence(n, world):
    got = [shard_range(n, r, world) for r in range(world)]
    assert got[0][0] == 0 and got[-1][1] == n
    sizes = [hi - lo for lo, hi in got]
    assert all(a[1] == b[0] for a, b in zip(got, got[1:]))
    assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(n, world, world)


# ---------------------------------------------------------------- synthetic data
def test_synth_is_deterministic_and_well_formed():
    a = synth.make_frames(3, 64, 48, seed=3)
    b = synth.make_frames(3, 64, 48, seed=3)
    c = synth.make_frames(3, 64, 48, seed=4)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert not np.array_equal(a[0], c[0])
    color, pos, edge = a
    assert color.shape == (3, 64, 48, 4) and pos.shape == (3, 64, 48, 4) and edge.shape == (3, 64, 48)
    cover = (color[..., 3] > 0).mean()
    assert 0.1 < cover < 0.8
    assert np.all(color[color[..., 3] == 0][:, :3] == 0)
    assert set(np.unique(edge)) <= {0, 255} and 0 < (edge == 0).mean() < 0.2
    sd_a, sd_b = synth.make_state_dict(1, seed=8), synth.make_state_dict(1, seed=8)
    assert all(np.array_equal(sd_a[k], sd_b[k]) for k in sd_a)


def test_algorithmic_flop_model_matches_baseline_md():
    # BASELINE.md section 3: MAC per full-resolution pixel, stage 1 live = 567552, stage 2 = 1037056
    def macs(stage):
        f, cin, k0 = [32, 64, 128, 128, 128, 64], 6, (3 if stage == 1 else 7)
        m = k0 * k0 * cin * f[0] + 9 * f[0] * f[1] / 4 + 9 * f[1] * f[2] / 16 + 14 * 9 * f[2] * f[2] / 16
        m += 9 * (f[3] + f[2]) * f[4] / 4 + 9 * (f[4] + f[1]) * f[4] + k0 * k0 * (f[0] + f[4] + cin) * f[5]
        m += (2 if stage == 2 else 1) * 9 * f[5] * f[5] + 3 * f[5]
        return m
    assert macs(1) == 567552 and macs(2) == 1037056


def test_subpixel_decomposition_of_upsample_conv_is_exact():
    """The sub-pixel plan of stage 2 (default; engine.cu compile_layer / conv_halo_persist_kernel<true>) replaces
    nearest-x2 + 3x3 conv (models.py:180-192) by four 2x2 convolutions on the low-resolution tensor.  Same index
    arithmetic restated with torch: class (py, px) writes out[2y+py, 2x+px], tap (a, b) reads in[y+a-1+py, x+b-1+px]
    with the 3x3 weights that hit that source pixel summed - equal to the reference composition including the border."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 5, 7, 6, generator=g, dtype=torch.float64)
    w = torch.randn(4, 5, 3, 3, generator=g, dtype=torch.float64)
    want = F.conv2d(F.interpolate(x, scale_factor=2, mode="nearest"), w, padding=1)

    def members(parity, tap):
        if parity == 0:
            return (0, 0) if tap == 0 else (1, 2)
        return (0, 1) if tap == 0 else (2, 2)

    got = torch.zeros_like(want)
    for py in range(2):
        for px in range(2):
            wc = torch.zeros(4, 5, 2, 2, dtype=torch.float64)
            for a in range(2):
                for b in range(2):
                    r0, r1 = members(py, a)
                    c0, c1 = members(px, b)
                    wc[:, :, a, b] = w[:, :, r0:r1 + 1, c0:c1 + 1].sum(dim=(2, 3))
            # asymmetric zero padding: (1 - py) rows above, py below; (1 - px) columns left, px right
            xp = F.pad(x, (1 - px, px, 1 - py, py))
            got[:, :, py::2, px::2] = F.conv2d(xp, wc)
    assert torch.allclose(got, want, rtol=0, atol=1e-12)


def test_n128_issue_form_of_the_split_fp16_product():
    """Split-fp16 conv_11 (engine.cu compile_layer, ConvParams::n128): the weight tile of a (tap, 32-channel block) is a
    no-swizzle K-major tile of 128 rows [W_hi ; W_lo] x 32 channels; a_hi x tile is one N = 128 MMA, a_lo x (first 64 rows) one
    N = 64 MMA, and the epilogue adds columns c and 64 + c.  Restated with numpy: (1) the byte offset formula tiles the 8 KB
    tile exactly once, (2) the two-MMA form equals a_hi.W_hi + a_lo.W_hi + a_hi.W_lo, (3) which is within 2^-20 relative of
    the fp32 product (the lo x lo term is the only thing dropped)."""
    rng = np.random.default_rng(7)
    offs = set()
    for row in range(128):
        for c in range(32):
            offs.add((row // 8) * 512 + (c // 8) * 128 + (row % 8) * 16 + (c % 8) * 2)
    assert len(offs) == 128 * 32 and min(offs) == 0 and max(offs) == 8190 and all(o % 2 == 0 for o in offs)

    a = rng.standard_normal((128, 32)).astype(np.float32) * 3
    w = rng.standard_normal((64, 32)).astype(np.float32)
    a_hi = a.astype(np.float16); a_lo = (a - a_hi.astype(np.float32)).astype(np.float16)
    w_hi = w.astype(np.float16); w_lo = (w - w_hi.astype(np.float32)).astype(np.float16)
    f = lambda t: t.astype(np.float64)
    tile = np.concatenate([f(w_hi), f(w_lo)], axis=0)                  # 128 rows
    d = f(a_hi) @ tile.T                                               # N = 128: [hi.W_hi | hi.W_lo]
    d[:, :64] += f(a_lo) @ tile[:64].T                                 # N = 64 on the first 64 rows
    got = d[:, :64] + d[:, 64:]                                        # epilogue: K-split sum, stride 64
    three = f(a_hi) @ f(w_hi).T + f(a_lo) @ f(w_hi).T + f(a_hi) @ f(w_lo).T
    assert np.allclose(got, three, rtol=0, atol=1e-12)
    exact = f(a) @ f(w).T
    assert np.abs(got - exact).max() < 2.0 ** -20 * np.abs(f(a)).max() * np.abs(f(w)).max() * 32


def test_work_assignment_properties():
    """shard_range / assign_work (pipeline.py, SURVEY 8e) over many job shapes: the shares are contiguous, ordered, differ by at
    most one frame, and tile the clip exactly; characters land on exactly one rank each."""
    from hypothesis import given, settings, strategies as st
    from drawingspinup_b200.pipeline import assign_work, shard_range

    @settings(max_examples=200, deadline=None)
    @given(st.integers(0, 5000), st.integers(1, 64))
    def frames(n, world):
        spans = [shard_range(n, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [hi - lo for lo, hi in spans]
        assert max(sizes) - min(sizes) <= 1 and sizes == sorted(sizes, reverse=True)
        assert [assign_work(n, 1, r, world) for r in range(world)] == [{0: s} for s in sizes]

    @settings(max_examples=200, deadline=None)
    @given(st.integers(2, 40), st.integers(1, 64), st.integers(0, 300))
    def characters(n_chars, world, per_char):
        shares = [assign_work(n_chars * per_char, n_chars, r, world) for r in range(world)]
        owners = sorted(c for s in shares for c in s)
        assert owners == list(range(n_chars)) and all(v == per_char for s in shares for v in s.values())
        assert max(len(s) for s in shares) - min(len(s) for s in shares) <= 1

    frames()
    characters()
