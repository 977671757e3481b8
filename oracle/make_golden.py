"""TEST INFRASTRUCTURE ONLY - mint golden fixtures from the LIVE reference.

Run in the build container (needs /root/reference, read-only; never at test time):

    python oracle/make_golden.py

Imports the unmodified reference modules from ``/root/reference/3_style_translator`` and stores
small input/output vectors under ``tests/golden/`` so that the oracle port - and through it the
CUDA path - stays pinned to the reference on boxes where the reference is absent.  The reference
ships no golden vectors of its own (SURVEY.md 8c), so these are the pins.

What is recorded (all seeded, see drawingspinup_b200/synth.py):
  * ``GeneratorJ_RIC.forward`` / ``GeneratorJ.forward`` outputs (training/models.py:293-356, 113-129)
    on 2 synthetic frames at 32x40, default YAML configuration, synthetic state dicts;
  * ``generate_coordinates`` (models.py:551-604, its ``.cuda()`` neutralised) at 24x20;
  * ``DatasetFullImages.__getitem__`` (data.py:23-47) incl. the stage-2 edge burn-in, via real PNGs;
  * ``to_image_space`` (custom_transforms.py:7-8) known answers;
  * ``pos2edge`` (run_render.py:31-57; the function is extracted with ``ast`` because importing the
    module needs Blender-side packages);
  * the state-dict layout (keys in order, shapes, dtypes) of the models ``build_model`` (trainers.py:33-35)
    makes for both stages, and the PNG frames the unmodified ``test_stage1.py`` / ``test_stage2.py`` write
    for a synthetic 3-frame character (``GOLDEN_ONLY=scripts`` records just these two files).
"""
from __future__ import annotations

import ast
import os
import sys
import tempfile
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference/3_style_translator"
OUT = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)
warnings.filterwarnings("ignore")

from drawingspinup_b200 import synth  # noqa: E402

ARGS = dict(use_bias=False, tanh=True, append_smoothers=True, resnet_blocks=7,
            filters=[32, 64, 128, 128, 128, 64], input_channels=6)


def _no_cuda(fn, *a, **k):
    """Run ``fn`` with torch.Tensor.cuda turned into the identity (models.py:602 is unconditional)."""
    orig = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *aa, **kk: self
    try:
        return fn(*a, **k)
    finally:
        torch.Tensor.cuda = orig


def reference_scripts():
    """Layout of the models ``build_model`` returns, and one run of the unmodified stage-1 and stage-2 scripts on the
    CPU (the YAML's ``device: cuda:0`` is replaced by ``cpu`` as the configs are read) over a synthetic character whose
    checkpoints are ``synth.make_state_dict(stage, out_gain=0.25)``.  Stage 2 reads the PNGs stage 1 wrote."""
    import json
    import runpy
    import yaml
    from PIL import Image
    import training.trainers as rt
    layout = {}
    for name in ("GeneratorJ_RIC", "GeneratorJ"):
        sd = rt.build_model(name, dict(ARGS), "cpu").state_dict()
        layout[name] = [[k, list(v.shape), str(v.dtype)] for k, v in sd.items()]
    with open(os.path.join(OUT, "reference_state_dict_layout.json"), "w") as f:
        json.dump({"args": ARGS, "models": layout}, f, indent=0)

    uid, action, n, h, w, out_gain = "synthetic0001", "dab", 3, 64, 48, 0.25
    sds = tuple(synth.to_torch_state_dict(synth.make_state_dict(s, out_gain=out_gain)) for s in (1, 2))
    real_load, cwd, argv = yaml.load, os.getcwd(), list(sys.argv)

    def cpu_config(stream, Loader):
        cfg = real_load(stream, Loader=Loader)
        cfg["job"]["device"] = "cpu"
        return cfg

    with tempfile.TemporaryDirectory() as tmp:
        work = os.path.join(tmp, "3_style_translator")
        os.makedirs(work)
        for name in ("test_stage1.py", "test_stage2.py", "training", "configs"):
            os.symlink(os.path.join(REF, name), os.path.join(work, name))
        root = os.path.join(tmp, "dataset", "AnimatedDrawings", "preprocessed")     # config_stage1.yaml root_dir
        color, pos, edge = synth.write_character_tree(root, uid, {action: n}, h, w, seed=5, state_dicts=sds)[action]
        yaml.load = cpu_config
        try:
            os.chdir(work)
            for script in ("test_stage1.py", "test_stage2.py"):
                sys.argv = [script, "--uid", uid]
                _no_cuda(runpy.run_path, os.path.join(work, script), run_name="__main__")
        finally:
            yaml.load, sys.argv = real_load, argv
            os.chdir(cwd)
        base = os.path.join(root, uid, "mesh", "blender_render", action)
        res = {d: np.stack([np.array(Image.open(os.path.join(base, d, "%04d.png" % i))) for i in range(n)])
               for d in ("res_stage1_mask_pos", "res_stage2_mask_pos_edge")}
    np.savez_compressed(os.path.join(OUT, "reference_scripts.npz"), color=color, pos=pos, edge=edge,
                        stage1=res["res_stage1_mask_pos"], stage2=res["res_stage2_mask_pos_edge"],
                        out_gain=np.array(out_gain))
    print("reference script frames", {k: v.shape for k, v in res.items()})


def main():
    if os.environ.get("GOLDEN_ONLY", "") == "scripts":
        os.makedirs(OUT, exist_ok=True)
        return reference_scripts()
    import training.models as rm
    from training.data import DatasetFullImages
    from training.custom_transforms import to_image_space
    from PIL import Image
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)          # one summation order for the recorded vectors
    if os.environ.get("GOLDEN_ONLY", "") == "norm":      # add the norm-variant vectors without rewriting the older files
        real_save = np.savez_compressed
        np.savez_compressed = lambda path, **kw: real_save(path, **kw) if ("_norm_" in path) else None
    h, w, b = 32, 40, 2
    color, pos, edge = synth.make_frames(b, h, w, seed=101)

    # ---- dataset transform through real PNG files (data.py:23-47)
    with tempfile.TemporaryDirectory() as tmp:
        for sub in ("color", "pos", "edge"):
            os.makedirs(os.path.join(tmp, sub))
        for i in range(b):
            Image.fromarray(color[i]).save(os.path.join(tmp, "color", "%04d.png" % i))
            Image.fromarray(pos[i]).save(os.path.join(tmp, "pos", "%04d.png" % i))
            Image.fromarray(edge[i]).save(os.path.join(tmp, "edge", "%04d.png" % i))
        ds1 = DatasetFullImages(tmp, "color", True, True, False)
        ds2 = DatasetFullImages(tmp, "color", True, True, True)
        pre1 = np.stack([ds1[i]["pre"].numpy() for i in range(b)])
        pre2 = np.stack([ds2[i]["pre"].numpy() for i in range(b)])
        mask = np.stack([ds1[i]["pre_mask"].numpy() for i in range(b)])
    np.savez_compressed(os.path.join(OUT, "dataset_transform.npz"), color=color, pos=pos, edge=edge,
                        pre_stage1=pre1, pre_stage2=pre2, pre_mask=mask)

    # ---- generators
    for stage, cls, pre in ((1, rm.GeneratorJ_RIC, pre1), (2, rm.GeneratorJ, pre2)):
        sd_np = synth.make_state_dict(stage, seed=1234, out_gain=0.25)
        m = cls(**ARGS).eval()
        m.load_state_dict(synth.to_torch_state_dict(sd_np))
        with torch.no_grad():
            y = _no_cuda(m, torch.from_numpy(pre))
        np.savez_compressed(os.path.join(OUT, "generator_stage%d.npz" % stage), x=pre, y=y.numpy(),
                            seed=np.array(1234), out_gain=np.array(0.25))
        print("stage", stage, "y range", float(y.min()), float(y.max()))

    # ---- variant configuration: biases, no tanh, no smoothers, 2 blocks, wider filters, 5 input channels
    var = dict(use_bias=True, tanh=False, append_smoothers=False, resnet_blocks=2,
               filters=[64, 64, 128, 128, 64, 32], input_channels=5)
    xv = torch.from_numpy(np.random.default_rng(5).standard_normal((1, 5, 24, 32)).astype(np.float32))
    for stage, cls in ((1, rm.GeneratorJ_RIC), (2, rm.GeneratorJ)):
        sd_np = synth.make_state_dict(stage, seed=77, filters=var["filters"], resnet_blocks=2, input_channels=5,
                                      tanh=False, append_smoothers=False, use_bias=True, out_gain=0.25)
        m = cls(**var).eval()
        m.load_state_dict(synth.to_torch_state_dict(sd_np))
        with torch.no_grad():
            y = _no_cuda(m, xv)
        np.savez_compressed(os.path.join(OUT, "generator_variant_stage%d.npz" % stage), x=xv.numpy(), y=y.numpy())

    # ---- norm_layer='instance_norm' (models.py:34-35) and norm_layer=None, default widths, 2 residual blocks
    if os.environ.get("GOLDEN_ONLY", "") in ("", "norm"):
        xn = torch.from_numpy(pre2[:, :, :24, :32].copy())
        for norm in ("instance_norm", None):
            nv = dict(ARGS, resnet_blocks=2, norm_layer=norm)
            for stage, cls in ((1, rm.GeneratorJ_RIC), (2, rm.GeneratorJ)):
                if norm is None and stage == 1:
                    continue        # the reference's stage-1 forward indexes self.conv0[2] (models.py:303): IndexError without a norm module
                sd_np = synth.make_state_dict(stage, seed=91, resnet_blocks=2, out_gain=0.25, norm=norm or "none")
                m = cls(**nv).eval()
                m.load_state_dict(synth.to_torch_state_dict(sd_np))
                with torch.no_grad():
                    y = _no_cuda(m, xn)
                np.savez_compressed(os.path.join(OUT, "generator_%s_stage%d.npz" % (norm or "no_norm", stage)), x=xn.numpy(), y=y.numpy())
                print(norm, "stage", stage, "y range", float(y.min()), float(y.max()))
    if os.environ.get("GOLDEN_ONLY", "") == "norm":
        return

    # ---- RIC coordinates
    coords = _no_cuda(rm.generate_coordinates, 2, 24, 20)
    np.savez_compressed(os.path.join(OUT, "ric_coords_24x20.npz"), coords=coords[0].numpy())

    # ---- to_image_space known answers (SURVEY 8c KAT v) + random
    kat_in = np.array([-2, -1, -.5, 0, .0039, .5, .999, 1, 3], np.float32)
    rnd = np.random.default_rng(3).uniform(-1.2, 1.2, 4096).astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "to_image_space.npz"), kat_in=kat_in, kat_out=to_image_space(kat_in),
                        rnd_in=rnd, rnd_out=to_image_space(rnd))

    # ---- pos2edge (run_render.py:31-57), extracted without importing the Blender-side module
    import cv2
    src = open(os.path.join(REF, "run_render.py")).read()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "pos2edge"][0]
    ns = {"cv2": cv2, "np": np}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "run_render.py", "exec"), ns)
    c64, p64, _ = synth.make_frames(2, 64, 72, seed=9)
    edges = []
    with tempfile.TemporaryDirectory() as tmp:
        for i in range(2):
            path = os.path.join(tmp, "p%d.png" % i)
            cv2.imwrite(path, p64[i][..., [2, 1, 0, 3]])       # RGBA array -> BGRA file order
            edges.append(ns["pos2edge"](path))
    np.savez_compressed(os.path.join(OUT, "pos2edge.npz"), pos=p64, edges=np.stack(edges))
    reference_scripts()
    print("golden fixtures written to", OUT)


if __name__ == "__main__":
    main()
