"""B2 / `editany_nogradio.py` "runs unchanged" (BASELINE.json north_star):
  * `from_pretrained` (editany_lora.py:352-377) loads diffusers-layout checkpoints into the engines - the packed
    weights equal those packed from the same ldm state dict directly;
  * the reference's OWN entry script (read from /root/reference at test time, not copied) runs unmodified through
    `python -m editanything_b200.compat.run` semantics against synthetic test-sized checkpoints: model build ->
    `model.process(*input_data["args"], **input_data["kwargs"])` -> (refined, output, ref, text).
The operators are the CPU emulation (tests/cpu_ops.py) through the `_backend.OPS` seam; the same flow on CUDA is
tests/test_gpu_app.py / test_gpu_nogradio.py."""
import os
import pickle

import numpy as np
import pytest
import torch
from PIL import Image

from editanything_b200 import _backend
from editanything_b200.sam_spec import SAM_TINY
from editanything_b200.unet_spec import TINY
from editanything_b200.vae_spec import VaeConfig
from tests import cpu_ops, synth_ckpt
from tests.test_app_cpu import _inputs

REF = os.environ.get("EA_REFERENCE_ROOT", "/root/reference")
VCFG = VaeConfig(ch=64, ch_mult=(1, 1, 1, 1), num_res_blocks=1)
SCRIPT = '''import pickle
from editany_lora import EditAnythingLoraModel
model = EditAnythingLoraModel(
    base_model_path="runwayml/stable-diffusion-v1-5",
    controlmodel_name='LAION Pretrained(v0-4)-SD15',
    lora_model_path=None, use_blip=False, extra_inpaint=True,
)
with open('input_data.pkl', 'rb') as f:
    input_data = pickle.load(f)
refined, output, ref, text = model.process(*input_data['args'], **input_data['kwargs'])
'''     # this repo's wording of the reference's 15-line entry script (used where /root/reference is absent)


@pytest.fixture
def cpu_backend(monkeypatch):
    # the constructors place engines on cuda:0 whenever a GPU is present; the emulated operators work on CPU tensors
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    _backend.OPS = cpu_ops
    yield
    _backend.OPS = None


def make_model_root(root):
    """The four checkpoints editany_nogradio.py's constructor downloads (editany_lora.py:72-79,360,393), test-sized."""
    base = os.path.join(root, "runwayml", "stable-diffusion-v1-5")
    usd, vsd = synth_ckpt.write_pipeline(base, TINY, VCFG, seed=51)
    cns = {}
    for name, seed in (("shgao/edit-anything-v0-4-sd15", 52), ("lllyasviel/control_v11p_sd15_inpaint", 53),
                       ("lllyasviel/control_v11f1e_sd15_tile", 54)):
        cns[name] = synth_ckpt.write_unet_like(os.path.join(root, *name.split("/")), TINY, "controlnet", seed)
    return usd, vsd, cns


def test_from_pretrained_loads_the_same_weights(tmp_path, monkeypatch, cpu_backend):
    from editanything_b200.loading import ControlNetModel, ControlNetModel2
    from editanything_b200.nets import PackedNet
    from editanything_b200.pipeline import StableDiffusionControlNetInpaintPipeline
    usd, vsd, cns = make_model_root(str(tmp_path))
    monkeypatch.setenv("EA_MODEL_ROOT", str(tmp_path))
    cn = [ControlNetModel2.from_pretrained("shgao/edit-anything-v0-4-sd15", torch_dtype=torch.float16),
          ControlNetModel.from_pretrained("lllyasviel/control_v11p_sd15_inpaint", torch_dtype=torch.float16)]
    assert cn[0].cfg == cn[1].cfg and cn[0].cfg.model_channels == TINY.model_channels and cn[0].cfg.context_dim == TINY.context_dim
    pipe = StableDiffusionControlNetInpaintPipeline.from_pretrained("runwayml/stable-diffusion-v1-5", controlnet=cn,
                                                                   torch_dtype=torch.float16, safety_checker=None)
    dev = pipe.engine.dev
    ref_unet = PackedNet(pipe.engine.cfg, "unet", usd, dev)
    for k, v in ref_unet.w.items():
        assert torch.equal(v, pipe.engine.unet.w[k]), k
    ref_cn = PackedNet(pipe.engine.cfg, "controlnet", cns["lllyasviel/control_v11p_sd15_inpaint"], dev)
    for k, v in ref_cn.w.items():
        assert torch.equal(v, pipe.engine.cns[1].w[k]), k
    assert len(pipe.controlnet.nets) == 2 and pipe.vae_scale_factor == 8 and pipe.tokenizer.model_max_length == 16
    assert pipe.text_encoder.config.hidden_size == TINY.context_dim
    # the tile pipeline shares the packed UNet / VAE / text encoder of the first one (editany_lora.py:391-423)
    tile = StableDiffusionControlNetInpaintPipeline.from_pretrained(
        "runwayml/stable-diffusion-v1-5", controlnet=ControlNetModel2.from_pretrained("lllyasviel/control_v11f1e_sd15_tile"),
        torch_dtype=torch.float16, safety_checker=None, share_with=pipe)
    assert tile.engine.unet is pipe.engine.unet and tile.vae is pipe.vae and tile.text_encoder is pipe.text_encoder
    with pytest.raises(FileNotFoundError):
        ControlNetModel.from_pretrained("nobody/nothing")
    with pytest.raises(NotImplementedError):
        pipe.load_textual_inversion("x")


@pytest.mark.parametrize("source", ["reference", "own"])
def test_entry_script_runs_unchanged(source, tmp_path, monkeypatch, cpu_backend):
    from editanything_b200.compat.run import run_script
    if source == "reference":
        script = os.path.join(REF, "editany_nogradio.py")
        if not os.path.isfile(script):
            pytest.skip("reference tree not present")
    else:
        script = str(tmp_path / "nogradio_equivalent.py")
        open(script, "w").write(SCRIPT)
    make_model_root(str(tmp_path / "hub"))
    monkeypatch.setenv("EA_MODEL_ROOT", str(tmp_path / "hub"))
    work = tmp_path / "work"
    work.mkdir()
    monkeypatch.chdir(work)
    synth_ckpt.write_sam(str(work / "models" / "sam_vit_h_4b8939.pth"), SAM_TINY)       # editany_lora.py:54,85
    from editanything_b200.segment_anything import amg
    monkeypatch.setattr(amg.SamAutomaticMaskGenerator.__init__, "__defaults__",
                        (8, 64, -1e9, -1.0, 1.0, 0.7, 0, 0.7, 512 / 1500, 1, None, 0, "binary_mask"))   # random weights: keep every mask
    args, kwargs = _inputs()
    args = args[:8] + (64, 256, 20) + args[11:]          # detect at the tiny SAM's 256, 20 UniPC steps
    with open("input_data.pkl", "wb") as f:
        pickle.dump({"args": args, "kwargs": kwargs}, f)
    g = run_script(script)
    assert g["model"].__class__.__name__ == "EditAnythingLoraModel"
    refined, output, ref, text = g["refined"], g["output"], g["ref"], g["text"]
    assert text == args[5] and len(output) == 2 and len(refined) == 2
    assert all(isinstance(i, Image.Image) and i.size == (64, 64) for i in output)
    assert all(isinstance(i, Image.Image) and i.size == (128, 128) for i in refined)
    assert isinstance(ref[0], Image.Image) and np.array(ref[1]).max() == 255
    assert g["model"].tile_pipe.engine.unet is g["model"].pipe.engine.unet
    from editanything_b200.schedulers import UniPCMultistepScheduler
    assert isinstance(g["model"].pipe.scheduler, UniPCMultistepScheduler)
