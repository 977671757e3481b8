"""GPU (-m gpu): the CUDA path, called through the C ABI via the Python mirror classes, against the
CPU oracle and the golden vectors minted from the live reference.

Tolerances: fp32 outputs within 1e-3 max-abs (BASELINE.json north_star) in the parity-grade fp16x3
mode; the single-pass fp16 mode is checked against its documented error bound; uint8 steps are
bit-exact on identical fp32 inputs.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import DEFAULT_ARGS, VARIANT_ARGS
import drawingspinup_b200 as dsu
from drawingspinup_b200 import capi, synth
from oracle import reference_port as rp

pytestmark = pytest.mark.gpu
TOL = 1e-3            # north_star: max-abs fp32 vs the reference forward
TOL_FP16 = 2.5e-2     # single-pass fp16 operands on the (deliberately sensitive) synthetic weights


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _model(stage, dev, precision="fp16x3", args=None, seed=1234, deterministic=False, **sd_kw):
    a = dict(DEFAULT_ARGS if args is None else args)
    cls = dsu.GeneratorJ_RIC if stage == 1 else dsu.GeneratorJ
    sd = synth.to_torch_state_dict(synth.make_state_dict(
        stage, seed=seed, filters=a["filters"], resnet_blocks=a["resnet_blocks"], input_channels=a["input_channels"],
        tanh=a["tanh"], append_smoothers=a["append_smoothers"], use_bias=a["use_bias"], out_gain=0.25, **sd_kw))
    m = cls(precision=precision, deterministic=deterministic, **a)
    m.load_state_dict(sd)
    return m.to(dev).eval(), sd


def _oracle(stage, sd, x, args=None):
    a = DEFAULT_ARGS if args is None else args
    cfg = dict(rp.default_config(stage), **{k: a[k] for k in ("resnet_blocks", "tanh", "append_smoothers", "use_bias")})
    with torch.no_grad():
        if stage == 1:
            return rp.generator_j_ric_forward(sd, x, cfg, use_torchvision=True)
        return rp.generator_j_forward(sd, x, cfg)


def _frames_tensor(b, h, w, seed, stage):
    color, pos, edge = synth.make_frames(b, h, w, seed=seed)
    x = np.stack([rp.frame_to_tensor(color[i], pos[i], edge[i] if stage == 2 else None)[0] for i in range(b)])
    return torch.from_numpy(x)


# ------------------------------------------------------------------ whole-network parity
@pytest.mark.parametrize("stage", [1, 2])
@pytest.mark.parametrize("shape", [(2, 64, 48), (1, 72, 100), (3, 32, 32), (1, 4, 4), (2, 8, 12), (5, 20, 36)])
def test_forward_matches_oracle_fp16x3(dev, stage, shape):
    b, h, w = shape
    m, sd = _model(stage, dev)
    x = _frames_tensor(b, h, w, seed=h + w, stage=stage)
    with torch.no_grad():
        y = m(x.to(dev)).cpu()
    assert y.shape == (b, 3, h, w) and y.dtype == torch.float32
    assert (y - _oracle(stage, sd, x)).abs().max().item() < TOL


@pytest.mark.parametrize("stage", [1, 2])
def test_forward_matches_reference_golden(dev, golden_dir, stage):
    g = np.load(os.path.join(golden_dir, "generator_stage%d.npz" % stage))
    m, _ = _model(stage, dev, seed=int(g["seed"]))
    with torch.no_grad():
        y = m(torch.from_numpy(g["x"]).to(dev)).cpu().numpy()
    assert np.abs(y - g["y"]).max() < TOL


@pytest.mark.parametrize("stage", [1, 2])
def test_variant_configuration_matches_reference_golden(dev, golden_dir, stage):
    """use_bias=True, tanh=False, no smoothers, 2 blocks, other filters, 5 input channels."""
    g = np.load(os.path.join(golden_dir, "generator_variant_stage%d.npz" % stage))
    m, _ = _model(stage, dev, args=VARIANT_ARGS, seed=77)
    with torch.no_grad():
        y = m(torch.from_numpy(g["x"]).to(dev)).cpu().numpy()
    scale = max(1.0, float(np.abs(g["y"]).max()))       # no tanh: outputs are unbounded, tolerance relative to range
    assert np.abs(y - g["y"]).max() < TOL * scale


@pytest.mark.parametrize("stage", [1, 2])
def test_single_pass_fp16_error_bound(dev, stage):
    m, sd = _model(stage, dev, precision="fp16")
    x = _frames_tensor(2, 64, 64, seed=3, stage=stage)
    with torch.no_grad():
        y = m(x.to(dev)).cpu()
    err = (y - _oracle(stage, sd, x)).abs()
    assert err.max().item() < TOL_FP16 and err.mean().item() < 2e-3


@pytest.mark.parametrize("shape", [(1, 4, 4), (2, 20, 36), (3, 72, 100), (1, 132, 68)])
def test_first_layer_kernel_matches_tap_mode_and_oracle(dev, shape):
    """GeneratorJ.conv0 (models.py:44-46) in fp16 mode runs the im2col-free kernel (conv_first.cu: no-swizzle UMMA
    operand read from the halo tile); knob first=0 sends it through the tap-mode kernel.  Both compute the same fp16
    products with fp32 accumulation, so conv0 may differ by accumulation order only (<= 1 fp16 ulp of its range)."""
    b, h, w = shape
    m, sd = _model(2, dev, precision="fp16")
    x = _frames_tensor(b, h, w, seed=11, stage=2)
    out = {}
    for mode in ("0", "1"):
        m.set_knob("first", int(mode))
        with torch.no_grad():
            y = m(x.to(dev)).cpu()
        out[mode] = (y, m.debug_buffer(0, 0, (b, h, w, 40)).float()[..., :32])
    assert (out["0"][1] - out["1"][1]).abs().max().item() <= 2 ** -7       # conv0 activations (|v| < 8): one fp16 ulp
    ref = _oracle(2, sd, x)
    for mode in ("0", "1"):
        assert (out[mode][0] - ref).abs().max().item() < TOL_FP16


@pytest.mark.parametrize("width", [64, 128])
def test_first_layer_kernel_wider_outputs(dev, width):
    """filters[0] = 64 / 128: the first-layer kernel with 2 (resp. 1) K-split issuers and 4 (resp. 2) accumulator sets."""
    args = dict(DEFAULT_ARGS, filters=[width, 64, 128, 128, 128, 64], resnet_blocks=1)
    m, sd = _model(2, dev, precision="fp16", args=args)
    x = _frames_tensor(2, 40, 24, seed=5, stage=2)
    with torch.no_grad():
        y = m(x.to(dev)).cpu()
    err = (y - _oracle(2, sd, x, args)).abs()
    assert err.max().item() < TOL_FP16


@pytest.mark.parametrize("stage", [1, 2])
def test_nondefault_offsets_builtin_table(dev, stage):
    """The engine's own generate_coordinates restatement (no torch offsets supplied) also meets parity."""
    if stage == 2:
        pytest.skip("stage 2 has no RIC field")
    m, sd = _model(stage, dev)
    m._prepare_shape = lambda h, w: None          # do not hand torch's offsets to the engine
    x = _frames_tensor(1, 48, 64, seed=8, stage=stage)
    with torch.no_grad():
        y = m(x.to(dev)).cpu()
    assert (y - _oracle(stage, sd, x)).abs().max().item() < TOL


# ------------------------------------------------------------------ the benchmark size itself (BASELINE configs[1] / [2])
FP16_BOUND = 1e-2     # stated bound of the single-pass fp16 mode at 512x512 (measured 3-5e-3; the reference's own default GPU
                      # path - cuDNN TF32, the same 10-bit mantissa - sits at the same level, see bench.py gpu_baseline)
_ORACLE_CACHE = {}


def _oracle_cached(stage, size, seed):
    """One CPU-oracle forward per (stage, size): ~35 s for stage 1 at 512x512 on 8 cores, so it is shared by the
    fp16x3 and fp16 checks of the same frame."""
    key = (stage, size, seed)
    if key not in _ORACLE_CACHE:
        torch.set_num_threads(min(32, len(os.sched_getaffinity(0))))
        sd = synth.to_torch_state_dict(synth.make_state_dict(stage, seed=1234, out_gain=0.25))
        x = _frames_tensor(1, size, size, seed=seed, stage=stage)
        _ORACLE_CACHE[key] = (sd, x, _oracle(stage, sd, x))
    return _ORACLE_CACHE[key]


@pytest.mark.parametrize("stage,size", [(1, 512), (2, 512), (1, 528)])
def test_benchmark_size_parity(dev, stage, size):
    """One full-size frame against the CPU oracle: the RIC stencil tables of the 512 / 256 / 128 (and 528 / 264 / 132)
    levels, partial tiles and the persistent tile schedulers are exercised where bench.py measures.  fp16x3 (the mode
    bench.py reports as `value`) must meet the north_star's 1e-3; the fp16 mode is held to its stated bound."""
    sd, x, ref = _oracle_cached(stage, size, seed=40 + stage)
    errs = {}
    for prec in ("fp16x3", "fp16"):
        m, _ = _model(stage, dev, precision=prec)
        with torch.no_grad():
            y = m(x.to(dev)).cpu()
        errs[prec] = (y - ref).abs().max().item()
        del m
    print("stage %d %dx%d max|dy|: fp16x3 %.3e, fp16 %.3e" % (stage, size, size, errs["fp16x3"], errs["fp16"]))
    assert errs["fp16x3"] < TOL
    assert errs["fp16"] < FP16_BOUND


def test_reference_on_gpu_agrees_with_cpu_oracle(dev):
    """bench.py's parity gate checks the engine against the oracle port run on cuda with TF32 off; that checker itself is
    pinned to the CPU oracle here (same port code, torch's CUDA kernels instead of its CPU kernels)."""
    for stage in (1, 2):
        sd = synth.to_torch_state_dict(synth.make_state_dict(stage, seed=1234, out_gain=0.25))
        x = _frames_tensor(1, 96, 80, seed=9, stage=stage)
        ref = _oracle(stage, sd, x)
        old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
        try:
            sdd = {k: v.to(dev) for k, v in sd.items()}
            with torch.no_grad():
                y = (rp.generator_j_ric_forward(sdd, x.to(dev), use_torchvision=True) if stage == 1
                     else rp.generator_j_forward(sdd, x.to(dev))).cpu()
        finally:
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        assert (y - ref).abs().max().item() < 2e-5


@pytest.mark.parametrize("env", [{"DSU_N128": "0"}, {"DSU_N128": "1"}, {"DSU_FIRST": "0"}, {"DSU_N128": "1", "DSU_HALO_NSETS": "1"}])
def test_split_fp16_stage2_plan_variants(dev, env, monkeypatch):
    """Split-fp16 stage 2, plan-time variants (knobs read once at dsu_create): conv_11 / the smoothers with and without the
    N = 128 issue form ([W_hi ; W_lo] no-swizzle weight tiles, 128-column accumulators summed by the epilogue, one or two
    accumulator sets), conv0 in the im2col-free kernel with a lo plane or in tap mode.  All of them compute the same
    three fp16 product sums, so they agree to fp32 accumulation order and all meet the parity tolerance."""
    x = _frames_tensor(2, 72, 100, seed=29, stage=2)
    m0, sd = _model(2, dev)
    with torch.no_grad():
        y0 = m0(x.to(dev)).cpu()
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    m1, _ = _model(2, dev)
    with torch.no_grad():
        y1 = m1(x.to(dev)).cpu()
    ref = _oracle(2, sd, x)
    assert (y1 - y0).abs().max().item() < 1e-4
    assert (y0 - ref).abs().max().item() < TOL and (y1 - ref).abs().max().item() < TOL


# ------------------------------------------------------------------ norm_layer variants of the constructor (models.py:29-35)
def _norm_model(stage, dev, norm, precision="fp16x3", blocks=2, seed=91):
    cls = dsu.GeneratorJ_RIC if stage == 1 else dsu.GeneratorJ
    args = dict(DEFAULT_ARGS, resnet_blocks=blocks, norm_layer=norm)
    sd = synth.to_torch_state_dict(synth.make_state_dict(stage, seed=seed, resnet_blocks=blocks, out_gain=0.25, norm=norm or "none"))
    m = cls(precision=precision, **args)
    m.load_state_dict(sd)
    cfg = dict(rp.default_config(stage), resnet_blocks=blocks, norm=norm)
    return m.to(dev).eval(), sd, cfg


@pytest.mark.parametrize("norm,stage", [("instance_norm", 1), ("instance_norm", 2), (None, 2)])
def test_norm_layer_variants_match_reference_golden(dev, golden_dir, norm, stage):
    """nn.InstanceNorm2d (statistics per frame and channel over H x W, no state) between every convolution and its activation -
    the engine leaves the raw convolution output in an fp32 scratch buffer and normalises in a separate pass (frames.cu) -
    and norm_layer=None, against vectors recorded from the live reference."""
    g = np.load(os.path.join(golden_dir, "generator_%s_stage%d.npz" % (norm or "no_norm", stage)))
    m, _, _ = _norm_model(stage, dev, norm)
    with torch.no_grad():
        y = m(torch.from_numpy(g["x"]).to(dev)).cpu().numpy()
    assert np.abs(y - g["y"]).max() < TOL


@pytest.mark.parametrize("stage", [1, 2])
@pytest.mark.parametrize("shape", [(3, 72, 100), (1, 132, 68)])
def test_instance_norm_ragged_shapes_and_batch_independence(dev, stage, shape):
    b, h, w = shape
    m, sd, cfg = _norm_model(stage, dev, "instance_norm")
    x = _frames_tensor(b, h, w, seed=41, stage=stage)
    with torch.no_grad():
        y = m(x.to(dev)).cpu()
        ref = rp.generator_j_ric_forward(sd, x, cfg, use_torchvision=True) if stage == 1 else rp.generator_j_forward(sd, x, cfg)
        assert (y - ref).abs().max().item() < TOL
        y0 = m(x[:1].to(dev)).cpu()                       # statistics are per frame: a frame does not see its batch mates
    assert (y0 - y[:1]).abs().max().item() < 1e-4
    m16, _, _ = _norm_model(stage, dev, "instance_norm", precision="fp16")
    with torch.no_grad():
        y16 = m16(x.to(dev)).cpu()
    assert (y16 - ref).abs().max().item() < TOL_FP16


# ------------------------------------------------------------------ tensor-memory RIC kernel configurations
def test_tensor_memory_kernel_issuer_and_stage_knobs(dev):
    """The tensor-memory RIC kernel with 1 / 3 issuing warps and the minimum weight ring gives the same result as the default
    configuration up to fp32 accumulation order (several warps accumulate into one TMEM accumulator)."""
    m, sd = _model(1, dev)
    x = _frames_tensor(2, 72, 100, seed=23, stage=1).to(dev)
    ref = _oracle(1, sd, x.cpu())
    with torch.no_grad():
        y0 = m(x).cpu()
        for ni, sb in ((1, 2), (3, 2), (6, 4)):
            m.set_knob("tm_ni", ni)
            m.set_knob("tm_sb", sb)
            y = m(x).cpu()
            assert (y - y0).abs().max().item() < 1e-4
            assert (y - ref).abs().max().item() < TOL


# ------------------------------------------------------------------ size-independent properties at full size
@pytest.mark.parametrize("stage", [1, 2])
def test_batch_invariance_and_determinism_512(dev, stage):
    """Bit-reproducible in deterministic mode (stage 1: one issuing warp; stage 2 always).  The default stage-1 configuration
    lets six warps accumulate into one TMEM accumulator, so repeated runs agree to fp32 accumulation order only."""
    m, _ = _model(stage, dev, precision="fp16", deterministic=True)
    x = _frames_tensor(3, 512, 512, seed=21, stage=stage).to(dev)
    with torch.no_grad():
        full = m(x)
        again = m(x)
        one = m(x[1:2])
    assert torch.equal(full, again)                      # deterministic
    assert torch.equal(full[1:2], one)                   # KAT (vi): a frame does not depend on its batch
    assert torch.isfinite(full).all() and full.abs().max().item() <= 1.0
    if stage == 1:
        # default (six issuing warps) vs deterministic, in the parity-grade mode: accumulation-order noise only.  (In the fp16
        # mode a last-bit fp32 difference can flip an fp16 rounding of an activation, so two orders differ at that mode's own
        # error level, ~1e-3; both stay within its bound against the oracle.)
        det, _ = _model(stage, dev, precision="fp16x3", deterministic=True)
        fast, _ = _model(stage, dev, precision="fp16x3")
        with torch.no_grad():
            ref, a, b = det(x), fast(x), fast(x[1:2])
        assert (a - ref).abs().max().item() < 1e-4 and (a[1:2] - b).abs().max().item() < 1e-4


def test_frame_size_528_partial_tiles(dev):
    """KAT (vii): jumping's real frame size (blender_animation.py:70-77): 528/264/132 are not tile multiples."""
    m16, _ = _model(2, dev, precision="fp16")
    mx, sd = _model(2, dev, precision="fp16x3")
    x = _frames_tensor(1, 528, 528, seed=5, stage=2)
    with torch.no_grad():
        y = mx(x.to(dev)).cpu()
        y16 = m16(x.to(dev)).cpu()
    ref = _oracle(2, sd, x)
    assert (y - ref).abs().max().item() < TOL
    assert (y16 - ref).abs().max().item() < TOL_FP16


def test_stage1_dead_smoother_weights_do_not_matter(dev):
    """KAT (iii), models.py:348-352: conv_11_a.0 / .2 are loaded (strict keys) but never influence stage 1."""
    m, sd = _model(1, dev, deterministic=True)
    x = _frames_tensor(1, 48, 48, seed=2, stage=1).to(dev)
    with torch.no_grad():
        a = m(x)
        sd2 = dict(sd)
        sd2["conv_11_a.0.weight"] = torch.randn_like(sd["conv_11_a.0.weight"])
        sd2["conv_11_a.2.running_var"] = torch.rand_like(sd["conv_11_a.2.running_var"]) + 0.5
        m.load_state_dict(sd2)
        b = m(x)
    assert torch.equal(a, b)


def test_weight_reload_changes_output(dev):
    m, sd = _model(2, dev)
    x = _frames_tensor(1, 32, 32, seed=2, stage=2).to(dev)
    with torch.no_grad():
        a = m(x)
        sd2 = synth.to_torch_state_dict(synth.make_state_dict(2, seed=99, out_gain=0.25))
        m.load_state_dict(sd2)
        b = m(x).cpu()
    assert not torch.equal(a.cpu(), b)
    assert (b - _oracle(2, sd2, x.cpu())).abs().max().item() < TOL


def test_input_validation(dev):
    m, _ = _model(2, dev)
    with torch.no_grad():
        with pytest.raises(RuntimeError):
            m(torch.zeros(1, 5, 32, 32, device=dev))          # wrong channel count
        with pytest.raises(RuntimeError, match="multiples of 4"):
            m(torch.zeros(1, 6, 30, 32, device=dev))          # int(H/2), int(H/4) levels need H % 4 == 0
    m.train()
    with pytest.raises(RuntimeError, match="inference-only"):
        m(torch.zeros(1, 6, 32, 32, device=dev))


# ------------------------------------------------------------------ uint8 / frame steps: bit exact
def _ptr(t):
    return C.c_void_p(t.data_ptr())


def test_to_image_space_bit_exact(dev, golden_dir):
    g = np.load(os.path.join(golden_dir, "to_image_space.npz"))
    rng = np.random.default_rng(0)
    x = np.concatenate([g["kat_in"], g["rnd_in"], rng.uniform(-1.5, 1.5, 1 << 16).astype(np.float32),
                        (np.arange(-300, 300, dtype=np.float32) / 255.0)])
    xd = torch.from_numpy(x).to(dev)
    out = torch.empty(x.size, dtype=torch.uint8, device=dev)
    capi.check(capi.lib().dsu_to_image_space(_ptr(xd), _ptr(out), x.size, None), "to_image_space")
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), rp.to_image_space(x))
    assert list(out.cpu().numpy()[:9]) == [0, 0, 63, 127, 127, 191, 254, 255, 255]


def test_frames_to_tensor_bit_exact(dev, golden_dir):
    g = np.load(os.path.join(golden_dir, "dataset_transform.npz"))
    color, pos, edge = (torch.from_numpy(g[k]).to(dev) for k in ("color", "pos", "edge"))
    b, h, w, _ = color.shape
    for e, key in ((None, "pre_stage1"), (edge, "pre_stage2")):
        pre = torch.empty((b, 6, h, w), dtype=torch.float32, device=dev)
        mask = torch.empty((b, 1, h, w), dtype=torch.float32, device=dev)
        capi.check(capi.lib().dsu_frames_to_tensor(_ptr(color), _ptr(pos), _ptr(e) if e is not None else None,
                                                   b, h, w, _ptr(pre), _ptr(mask), None), "frames_to_tensor")
        torch.cuda.synchronize()
        assert np.array_equal(pre.cpu().numpy(), g[key])          # reference DatasetFullImages output
        assert np.array_equal(mask.cpu().numpy(), g["pre_mask"])


def test_overlap_edge_and_compose_bit_exact(dev):
    color, pos, edge = synth.make_frames(2, 40, 56, seed=4)
    rgba = torch.from_numpy(color).to(dev).clone()
    edge_d = torch.from_numpy(edge).to(dev)              # keep device tensors alive across the async launches
    capi.check(capi.lib().dsu_overlap_edge(_ptr(edge_d), _ptr(rgba), 2 * 40 * 56, None), "overlap")
    want = np.stack([rp.overlap_edge_on_img(edge[i], color[i]) for i in range(2)])
    assert np.array_equal(rgba.cpu().numpy(), want)
    rng = np.random.default_rng(1)
    y = rng.uniform(-1.3, 1.3, (2, 3, 40, 56)).astype(np.float32)
    mask = np.stack([rp.frame_to_tensor(color[i], pos[i])[1] for i in range(2)])
    out = torch.empty((2, 40, 56, 4), dtype=torch.uint8, device=dev)
    y_d, mask_d = torch.from_numpy(y).to(dev), torch.from_numpy(mask).to(dev)
    capi.check(capi.lib().dsu_compose_rgba(_ptr(y_d), _ptr(mask_d), 2, 40, 56, _ptr(out), None), "compose")
    want = np.stack([rp.compose_rgba(y[i], mask[i]) for i in range(2)])
    assert np.array_equal(out.cpu().numpy(), want)


def test_pos2edge_bit_exact(dev, golden_dir):
    g = np.load(os.path.join(golden_dir, "pos2edge.npz"))
    pos = torch.from_numpy(g["pos"]).to(dev)
    b, h, w, _ = pos.shape
    out = torch.empty((b, h, w), dtype=torch.uint8, device=dev)
    capi.check(capi.lib().dsu_pos2edge(_ptr(pos), b, h, w, _ptr(out), None), "pos2edge")
    assert np.array_equal(out.cpu().numpy(), g["edges"])          # the reference's own cv2 result
    _, pos2, _ = synth.make_frames(2, 96, 80, seed=12)
    out2 = torch.empty((2, 96, 80), dtype=torch.uint8, device=dev)
    pos2_d = torch.from_numpy(pos2).to(dev)
    capi.check(capi.lib().dsu_pos2edge(_ptr(pos2_d), 2, 96, 80, _ptr(out2), None), "pos2edge")
    assert np.array_equal(out2.cpu().numpy(), np.stack([rp.pos2edge(pos2[i]) for i in range(2)]))


# ------------------------------------------------------------------ fused frame path and the two-stage chain
def test_fused_frame_path_equals_unfused_steps(dev):
    """forward_frames == frames_to_tensor -> forward -> compose (bitwise: same kernels, same fp32 values)."""
    b, h, w = 2, 64, 48
    color, pos, edge = synth.make_frames(b, h, w, seed=6)
    for stage in (1, 2):
        m, sd = _model(stage, dev, deterministic=True)
        c, p = torch.from_numpy(color).to(dev), torch.from_numpy(pos).to(dev)
        e = torch.from_numpy(edge).to(dev) if stage == 2 else None
        with torch.no_grad():
            out, y = m.forward_frames(c, p, e, return_float=True)
            x = torch.from_numpy(np.stack([rp.frame_to_tensor(color[i], pos[i], edge[i] if stage == 2 else None)[0]
                                           for i in range(b)])).to(dev)
            y2 = m(x)
        assert torch.equal(y, y2)
        want = np.stack([rp.compose_rgba(y[i].cpu().numpy(), rp.frame_to_tensor(color[i], pos[i])[1]) for i in range(b)])
        assert np.array_equal(out.cpu().numpy(), want)


def test_two_stage_chain_against_oracle_chain(dev):
    """stage 1 -> uint8 -> edge burn-in -> stage 2 (test_stage1.py + test_stage2.py back to back)."""
    from drawingspinup_b200.pipeline import StylizationPipeline
    b, h, w = 2, 64, 64
    color, pos, edge = synth.make_frames(b, h, w, seed=13)
    sd1 = synth.to_torch_state_dict(synth.make_state_dict(1, out_gain=0.25))
    sd2 = synth.to_torch_state_dict(synth.make_state_dict(2, out_gain=0.25))
    pipe = StylizationPipeline(sd1, sd2, dev, precision="fp16x3", batch=2, deterministic=True)
    out2, out1 = pipe.run(torch.from_numpy(color).to(dev), torch.from_numpy(pos).to(dev),
                          torch.from_numpy(edge).to(dev), keep_stage1=True)
    out1, out2 = out1.cpu().numpy(), out2.cpu().numpy()
    with torch.no_grad():
        x1 = torch.from_numpy(np.stack([rp.frame_to_tensor(color[i], pos[i])[0] for i in range(b)]))
        y1 = rp.generator_j_ric_forward(sd1, x1, use_torchvision=True)
    want1 = np.stack([rp.compose_rgba(y1[i].numpy(), rp.frame_to_tensor(color[i], pos[i])[1]) for i in range(b)])
    d1 = np.abs(out1.astype(np.int32) - want1.astype(np.int32))
    assert d1.max() <= 1 and (d1 > 0).mean() < 0.01          # <=1 LSB where fp32 sits on an integer boundary
    assert np.array_equal(out1[..., 3], color[..., 3])        # alpha round trip is exact
    # stage 2 on the engine's own stage-1 bytes (what test_stage2.py would read back from disk)
    with torch.no_grad():
        x2 = torch.from_numpy(np.stack([rp.frame_to_tensor(out1[i], pos[i], edge[i])[0] for i in range(b)]))
        y2 = rp.generator_j_forward(sd2, x2)
    want2 = np.stack([rp.compose_rgba(y2[i].numpy(), rp.frame_to_tensor(out1[i], pos[i])[1]) for i in range(b)])
    d2 = np.abs(out2.astype(np.int32) - want2.astype(np.int32))
    assert d2.max() <= 1 and (d2 > 0).mean() < 0.01
    # host-buffer entry point gives the same bytes
    host_out = torch.empty((b, h, w, 4), dtype=torch.uint8).pin_memory()
    pipe.run_host(torch.from_numpy(color).pin_memory(), torch.from_numpy(pos).pin_memory(),
                  torch.from_numpy(edge).pin_memory(), host_out)
    assert np.array_equal(host_out.numpy(), out2)


def test_pipeline_derives_edges_from_pos(dev):
    """f1 (run_render.py:31-57, 117-120): with derive_edge the stage-2 ingest burns the edges it finds in the pos frames itself;
    the result equals the pipeline fed with the edge map the reference would have written (255 - pos2edge), bit for bit."""
    from drawingspinup_b200.pipeline import StylizationPipeline
    b, h, w = 2, 64, 80
    color, pos, _ = synth.make_frames(b, h, w, seed=29)
    edge = np.stack([255 - rp.pos2edge(pos[i]) for i in range(b)]).astype(np.uint8)
    assert (edge < 255).any()
    sd1 = synth.to_torch_state_dict(synth.make_state_dict(1, out_gain=0.25))
    sd2 = synth.to_torch_state_dict(synth.make_state_dict(2, out_gain=0.25))
    c_d, p_d, e_d = (torch.from_numpy(a).to(dev) for a in (color, pos, edge))
    given = StylizationPipeline(sd1, sd2, dev, precision="fp16x3", batch=2, deterministic=True).run(c_d, p_d, e_d)
    derived = StylizationPipeline(sd1, sd2, dev, precision="fp16x3", batch=2, deterministic=True, derive_edge=True).run(c_d, p_d, None)
    assert torch.equal(given, derived)


def test_c_abi_host_entry_point(dev):
    b, h, w = 1, 32, 48
    color, pos, edge = synth.make_frames(b, h, w, seed=17)
    m, _ = _model(2, dev)
    c, p, e = (torch.from_numpy(a).pin_memory() for a in (color, pos, edge))
    out = torch.empty((b, h, w, 4), dtype=torch.uint8).pin_memory()
    m.forward_frames_host(c, p, e, out, dev)
    with torch.no_grad():
        want = m.forward_frames(c.to(dev), p.to(dev), e.to(dev)).cpu()
    assert torch.equal(out, want)


def test_flop_model_and_launch_count(dev):
    m1, _ = _model(1, dev)
    m2, _ = _model(2, dev)
    assert abs(m1.algorithmic_flops(1, 512, 512) - 297.56e9) / 297.56e9 < 1e-3     # BASELINE.md section 3
    assert abs(m2.algorithmic_flops(1, 512, 512) - 543.72e9) / 543.72e9 < 1e-3
    # ingest + fused convs (+ RIC tap expansion of the input and 2 max-pools in stage 1; its dead smoother conv is not launched)
    # stage 1: ingest + 21 fused convolutions + 2 max-pools; stage 2: each nearest-x2 up-convolution is four sub-pixel launches
    assert m1.kernel_launches(1, 512, 512) == 1 + 21 + 2 and m2.kernel_launches(1, 512, 512) == 1 + 22 + 6


def test_profile_hook_reports_every_launch(dev):
    """dsu_profile_forward / dsu_step_name: one entry per launch after the ingest, FLOPs add up to the model's."""
    for stage in (1, 2):
        m, _ = _model(stage, dev, precision="fp16")
        x = _frames_tensor(1, 64, 64, seed=4, stage=stage).to(dev)
        with torch.no_grad():
            m(x)
        rows = m.profile_layers(1, 64, 64, reps=1)
        assert len(rows) == m.kernel_launches(1, 64, 64) - 1
        names = [r[0] for r in rows]
        assert names[-1] == "conv_11_a.3" and any(n.startswith("upconv1") for n in names) and ("maxpool" in names) == (stage == 1)
        assert all(ms > 0 for _, ms, _ in rows)
        assert abs(sum(f for _, _, f in rows) - m.algorithmic_flops(1, 64, 64)) / m.algorithmic_flops(1, 64, 64) < 1e-6


def test_multi_gpu_shard_equivalence(dev):
    """N-GPU frame sharding == single GPU, bitwise (SURVEY.md section 4 item 5)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from drawingspinup_b200.pipeline import StylizationPipeline, shard_range
    color, pos, edge = synth.make_frames(6, 64, 64, seed=31)
    sd1 = synth.to_torch_state_dict(synth.make_state_dict(1, out_gain=0.25))
    sd2 = synth.to_torch_state_dict(synth.make_state_dict(2, out_gain=0.25))
    outs = []
    single = None
    for r in range(2):
        d = torch.device("cuda", r)
        pipe = StylizationPipeline(sd1, sd2, d, precision="fp16", batch=4, deterministic=True)
        lo, hi = shard_range(6, r, 2)
        outs.append(pipe.run(*(torch.from_numpy(a[lo:hi]).to(d) for a in (color, pos, edge))).cpu())
        if r == 0:
            single = pipe.run(*(torch.from_numpy(a).to(d) for a in (color, pos, edge))).cpu()
    assert torch.equal(torch.cat(outs), single)


# ------------------------------------------------------------------ the reference scripts' frame loop on the engine
def test_engine_reproduces_reference_script_frames(dev, golden_dir, monkeypatch):
    """SURVEY.md section 4 item 4: the frames the unmodified test_stage1.py / test_stage2.py wrote for a synthetic 3-frame
    character on the reference's own models (recorded by oracle/make_golden.py) are what the engine gives in their place
    (<= 1 LSB).  The engine classes come from a ``training.models`` module rebound by install() and are built as
    build_model builds them (trainers.py:33-35); every frame then goes through the scripts' loop: dataset transform,
    forward, to_image_space, mask as alpha.  Stage 2 reads the stage-1 frames the reference wrote (config_stage2.yaml:61
    pre_dir), so both stages are compared on identical inputs."""
    import types
    g = np.load(os.path.join(golden_dir, "reference_scripts.npz"))
    color, pos, edge = g["color"], g["pos"], g["edge"]
    monkeypatch.setenv("DSU_PRECISION", "fp16x3")
    models = dsu.install(types.ModuleType("training.models"))
    for stage, name, pre, want in ((1, "GeneratorJ_RIC", color, g["stage1"]), (2, "GeneratorJ", g["stage1"], g["stage2"])):
        gen = getattr(models, name)(**DEFAULT_ARGS).to(dev)
        gen.load_state_dict(synth.to_torch_state_dict(synth.make_state_dict(stage, out_gain=float(g["out_gain"]))))
        gen.eval()
        got = []
        with torch.no_grad():
            for i in range(color.shape[0]):
                x, mask = rp.frame_to_tensor(pre[i], pos[i], edge[i] if stage == 2 else None)
                y = gen(torch.from_numpy(x)[None].to(dev))[0]
                got.append(rp.compose_rgba(y.cpu().numpy(), mask))
        d = np.abs(np.stack(got).astype(np.int32) - want.astype(np.int32))
        assert d.max() <= 1 and (d > 0).mean() < 0.01, (stage, d.max(), (d > 0).mean())
