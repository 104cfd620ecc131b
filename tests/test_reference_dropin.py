"""The drop-in, executed: the reference's own experiment script ``train_settings/dvd/val_TDiff.py`` is run with the three import
swaps of INTEGRATION.md (and nothing else changed) against synthetic checkpoints and a synthetic photo folder.

* CPU (build container): ``run(settings)`` goes through ``setup_dist`` -> ``create_model_and_diffusion`` -> the reference's
  preprocessing nets -> ``model.load_state_dict(..., strict=False)`` -> ``model.to(dev).eval()`` -> DataLoader ->
  ``run_evaluation_docunet(...)``; the evaluation call is intercepted (the product has no CPU path) and its arguments checked.
* GPU (``-m gpu``): the same script runs for real, and next to it the UNMODIFIED script with the reference's own model / sampler /
  unwarp on the same GPU, same seeds: the dewarped PNGs of the two runs must agree (PSNR >= 45 dB).

The two tests that execute val_TDiff.py skip when no reference tree is present.  The last test needs no reference tree: it runs the
same drop-in path on GPU and compares it with the reference's stored outputs in tests/golden/."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import ref_harness as RH

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_reference = pytest.mark.skipif(not RH.available(), reason="reference tree not present (baseline/_ref is created by __graft_entry__.build())")

SWAPS = [
    ("from .evaluation import run_evaluation_docunet",
     "from dvd_b200.evaluation import run_evaluation_docunet"),
    ("from .improved_diffusion import dist_util, logger",
     "from dvd_b200 import dist as dist_util\nfrom .improved_diffusion import logger"),
    ("from .improved_diffusion.script_util import (args_to_dict,\n                                             create_model_and_diffusion,\n"
     "                                             model_and_diffusion_defaults)",
     "from dvd_b200.script_util import args_to_dict, create_model_and_diffusion, model_and_diffusion_defaults"),
]


def _load_val_tdiff(patched: bool):
    """Imports val_TDiff.py from the reference tree as a module of the package train_settings.dvd (so that its relative imports
    work), optionally with the three import swaps of INTEGRATION.md applied to the source text."""
    RH._setup_path()
    import train_settings.dvd as pkg                                        # the reference package (namespace or regular)
    path = os.path.join(RH.REF_ROOT, "train_settings", "dvd", "val_TDiff.py")
    src = open(path).read()
    if patched:
        for old, new in SWAPS:
            assert old in src, f"val_TDiff.py no longer contains the import to swap: {old!r}"
            src = src.replace(old, new)
    name = "train_settings.dvd.val_TDiff_" + ("b200" if patched else "ref")
    mod = types.ModuleType(name)
    mod.__package__ = "train_settings.dvd"
    mod.__file__ = path
    sys.modules[name] = mod
    exec(compile(src, path, "exec"), mod.__dict__)
    return mod


def _make_workspace(tmp_path, n_docs=2, H=96, W=128):
    """Synthetic checkpoints (random-init reference modules + the synthetic DiT state dict) and a folder of synthetic photos."""
    import cv2
    import synth_workload as synth
    nets = RH.build_preprocessing_nets()
    ck = tmp_path / "checkpoints"
    ck.mkdir()
    torch.manual_seed(7)
    torch.save(synth.make_state_dict(1234), ck / "model1852000.pt")
    # reload_segmodel (geotr_core.py:1090-1110) strips a 6-character prefix from every key
    torch.save({"model." + k: v for k, v in nets["GeoTr_Seg_Inf"].msk.state_dict().items()}, ck / "seg.pth")
    torch.save({"model": nets["line UNet"].state_dict()}, ck / "line_model2.pth")
    torch.save({"model": nets["Seg(U2NETP)"].state_dict()}, ck / "seg_model.pth")
    data = tmp_path / "docs"
    data.mkdir()
    for i in range(n_docs):
        photo = synth.make_photo(H, W, 50 + i, "page")[0].permute(1, 2, 0).numpy().astype(np.uint8)
        cv2.imwrite(str(data / f"doc{i}.png"), photo[:, :, ::-1])
    return ck, data


def _settings(tmp_path, ck, data, name):
    RH._setup_path()
    import admin.settings as ws_settings
    s = ws_settings.Settings()
    s.name = name
    e = s.env
    e.eval_dataset_name, e.eval_dataset = "docunet", str(data)
    e.model_path = str(ck / "model1852000.pt")
    e.seg_model_path = str(ck / "seg.pth")
    e.line_seg_model_path = str(ck / "line_model2.pth")
    e.new_seg_model_path = str(ck / "seg_model.pth")
    return s


@needs_reference
def test_val_tdiff_with_swapped_imports_reaches_the_evaluation_call(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("MASTER_ADDR", "127.0.0.1")
    ck, data = _make_workspace(tmp_path)
    import dvd_b200.evaluation as EV
    from dvd_b200.model import DiT
    from dvd_b200.sampler import SpacedDiffusion
    from dvd_b200.weights import required_keys
    seen = {}

    def fake_eval(settings, logger, loader, diffusion, model, dewarp, line=None, seg=None):
        seen.update(settings=settings, loader=loader, diffusion=diffusion, model=model, dewarp=dewarp, line=line, seg=seg)

    monkeypatch.setattr(EV, "run_evaluation_docunet", fake_eval)
    mod = _load_val_tdiff(patched=True)
    assert mod.run_evaluation_docunet is fake_eval and mod.create_model_and_diffusion.__module__ == "dvd_b200.script_util"
    try:
        mod.run(_settings(tmp_path, ck, data, "dropin"))
    finally:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    assert isinstance(seen["model"], DiT) and isinstance(seen["diffusion"], SpacedDiffusion)
    assert seen["diffusion"].num_timesteps == 3 and seen["diffusion"].settings is seen["settings"]          # val_TDiff.py:52
    sd = seen["model"].state_dict()
    assert all(k in sd for k in required_keys()) and len(sd) >= 369                                          # the checkpoint was loaded
    assert type(seen["dewarp"]).__name__ == "GeoTr_Seg_Inf" and type(seen["seg"]).__name__ == "Seg" and type(seen["line"]).__name__ == "UNet"
    batch = next(iter(seen["loader"]))
    assert tuple(batch["source_image"].shape) == (1, 3, 512, 512) and tuple(batch["source_image_ori"].shape) == (1, 3, 96, 128)
    assert len(seen["loader"]) == 2


@needs_reference
@pytest.mark.gpu
def test_val_tdiff_dropin_matches_the_unmodified_script_on_gpu(tmp_path, monkeypatch):
    """Both scripts end to end on cuda:0 with the same seeds: reference model + sampler + grid_sample vs dvd_b200."""
    from PIL import Image
    import torch.distributed as dist
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("MASTER_ADDR", "127.0.0.1")
    monkeypatch.setenv("DVD_PRECISION", "bf16x3")
    ck, data = _make_workspace(tmp_path, n_docs=2, H=480, W=640)
    os.makedirs(tmp_path / "vis_hp" / "debug_vis", exist_ok=True)          # the reference's debug dumps (gaussian_diffusion.py:606,614)
    # evaluation.py:152 constructs a torchvision VGG16 with pretrained weights (a download) that the default config never uses
    import torchvision
    vgg16 = torchvision.models.vgg16
    monkeypatch.setattr(torchvision.models, "vgg16", lambda *a, **k: vgg16(weights=None))
    torch.backends.cudnn.allow_tf32 = False                                 # strict fp32 reference (default would run its convs in TF32)
    torch.backends.cuda.matmul.allow_tf32 = False
    outs = {}
    for patched in (False, True):
        mod = _load_val_tdiff(patched)
        name = "b200" if patched else "ref"
        torch.manual_seed(1234); torch.cuda.manual_seed_all(1234)
        try:
            mod.run(_settings(tmp_path, ck, data, name))
        finally:
            if dist.is_initialized():
                dist.destroy_process_group()
        d = tmp_path / "vis_hp" / "docunet" / name / "dewarped_pred"
        outs[name] = {f: np.asarray(Image.open(d / f)).astype(np.float64) for f in sorted(os.listdir(d))}
    assert sorted(outs["ref"]) == sorted(outs["b200"]) == ["warped_doc0.png", "warped_doc1.png"]
    for f in outs["ref"]:
        a, b = outs["ref"][f], outs["b200"][f]
        assert a.shape == b.shape == (480, 640, 3)
        mse = float(((a - b) ** 2).mean())
        psnr = 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)
        assert psnr >= 45.0, (f, psnr)


@pytest.mark.gpu
def test_dropin_evaluation_matches_reference_golden_on_gpu(golden_dir, tmp_path, monkeypatch):
    """What the drop-in side of val_TDiff.py runs, without the reference tree: create_model_and_diffusion with admin/local.py values,
    the full synthetic checkpoint loaded with strict=False, DVD_PRECISION=bf16x3, and run_evaluation_docunet over two documents
    with 480x640 photos.  The preprocessing nets are stand-ins that return each document's conditioning.  Each dewarped PNG must
    reach PSNR >= 45 dB against the unmodified reference's sampled map for that document (tests/golden/sample_S3_doc*.npz, same
    conditioning, weights and noise), unwarped by the oracle, which test_oracle_golden pins to the reference's own unwarp."""
    from PIL import Image
    import synth_workload as synth
    from oracle import dvd_oracle as O
    from dvd_b200.evaluation import run_evaluation_docunet
    from dvd_b200.script_util import args_to_dict, create_model_and_diffusion, model_and_diffusion_defaults
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("DVD_PRECISION", "bf16x3")
    dev = torch.device("cuda:0")

    class Env:      # admin/local.py values
        image_size = 64; num_channels = 128; num_res_blocks = 3; num_heads = 4; num_heads_upsample = -1
        attention_resolutions = "16,8"; dropout = 0.0; learn_sigma = False; sigma_small = False; class_cond = False
        diffusion_steps = 3; noise_schedule = "cosine"; timestep_respacing = ""; use_kl = False; predict_xstart = True
        rescale_timesteps = True; rescale_learned_sigmas = True; use_checkpoint = False; use_scale_shift_norm = True
        train_mode = "stage_1_dit_cross"; iter = True; use_gt_mask = False; use_line_mask = True; use_init_flow = False
        clip_denoised = False; n_batch = 2; time_variant = True; visualize = True; eval_dataset_name = "docunet"

    class Settings:
        env = Env(); name = "b200"

    model, diffusion = create_model_and_diffusion(**args_to_dict(Settings, model_and_diffusion_defaults().keys()), device=dev,
                                                  train_mode=Env.train_mode, tv=True)
    model.load_state_dict(synth.make_state_dict(1234), strict=False)
    model.to(dev).eval()
    assert model.precision == "bf16x3"
    # the golden maps were sampled from the 96x128 documents' conditioning; the full-resolution photo only enters the unwarp
    docs = [synth.make_doc_inputs(doc, H=96, W=128) for doc in (0, 1)]
    photos = [synth.make_photo(480, 640, 50 + doc, "page") for doc in (0, 1)]
    loader = [{"source_image": d["y512"], "source_image_ori": p, "path": [f"/data/doc{i}.png"]} for i, (d, p) in enumerate(zip(docs, photos))]
    cur = {}

    class Dewarp(torch.nn.Module):           # GeoTr_Seg_Inf stand-in, called first for every document: (ref_bm, mask_x)
        def forward(self, x):
            cur["doc"] = docs[len(cur.setdefault("seen", []))]
            cur["seen"].append(1)
            return torch.zeros(1, 2, 288, 288, device=x.device), cur["doc"]["mask_cat"].to(x.device)

    class Seg(torch.nn.Module):              # U2NETP stand-in: mskx, d0, hx6 .. hx1d (6 x 64 channels @ 64x64 -> 384)
        def forward(self, x):
            return (torch.zeros(1, 3, 288, 288, device=x.device), None) + tuple(cur["doc"]["mask_y512"].to(x.device).split(64, dim=1))

    class Line(torch.nn.Module):
        def forward(self, x):
            return cur["doc"]["line_msk"].to(x.device), None

    orig = diffusion.ddim_sample_loop          # the reference draws x_T on the host from seed 2000 + doc (make_doc_inputs)
    diffusion.ddim_sample_loop = lambda *a, **k: orig(*a, **{**k, "x_T": cur["doc"]["x_T"]})
    times = run_evaluation_docunet(Settings, None, loader, diffusion, model, Dewarp(), Line(), Seg())
    assert sorted(times) == [0, 1]
    for doc, photo in enumerate(photos):
        g = np.load(os.path.join(golden_dir, f"sample_S3_doc{doc}.npz"))
        ref = O.to_uint8_hwc(O.unwarp(torch.from_numpy(g["sample"]), photo)).astype(np.float64)
        png = np.asarray(Image.open(tmp_path / "vis_hp" / "docunet" / "b200" / "dewarped_pred" / f"warped_doc{doc}.png")).astype(np.float64)
        assert png.shape == ref.shape == (480, 640, 3)
        mse = float(((png - ref) ** 2).mean())
        psnr = 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)
        assert psnr >= 45.0, (doc, psnr)
