"""`EditAnythingLoraModel.process` (SURVEY.md §8b row B1, editanything_b200/app.py):
  1. against the REFERENCE's own `process` (the method's unmodified source, run with the pipelines replaced by
     spies by oracle/make_golden_ref.py, which records every call in tests/golden/ref_app_process.pt): both must hand
     the pipelines the same tensors, PIL images, scales, generator state - i.e. identical pre-processing, control
     map, inpaint condition, prompt windows, RNG consumption and tile-pass arguments - and return the same structure;
  2. end to end on synthetic tiny networks (engines on the CPU emulation of the operators), replaying an
     `input_data.pkl` synthesised the way the reference's decorator writes it (annotator/util.py:75-93)."""
import os
import pickle
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from PIL import Image

from editanything_b200 import app

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class _Ids(torch.Tensor):
    """input_ids that survive `.to("cuda")` on a CPU-only box."""
    @staticmethod
    def __new__(cls, data):
        return torch.Tensor._make_subclass(cls, data)

    def to(self, *a, **k):
        return self


class _Tok:
    model_max_length = 8

    def __call__(self, text, return_tensors="pt", truncation=False, padding=None, max_length=None):
        ids = [1] + [3 + (sum(map(ord, w)) % 50) for w in text.replace(",", " ").split()] + [2]
        if padding == "max_length" and max_length is not None:
            ids = ids + [0] * (max_length - len(ids))
        return SimpleNamespace(input_ids=_Ids(torch.tensor([ids])))


class _Enc(torch.nn.Module):
    def __init__(self, dim=64):
        super().__init__()
        torch.manual_seed(0)
        self.emb = torch.nn.Embedding(64, dim)

    def forward(self, ids):
        x = self.emb(torch.as_tensor(ids))
        return (x + x.cumsum(1) * 0.1,)


class SpyPipe:
    """Records every call; returns deterministic PIL images of the requested size."""
    def __init__(self):
        self.tokenizer, self.text_encoder, self.calls = _Tok(), _Enc(), []
        self._execution_device = torch.device("cpu")

    def __call__(self, **kw):
        gen = kw["generator"]
        kw["generator_state"] = gen.get_state().clone()
        draw = torch.rand(3, generator=gen)                      # consume the generator like a real pipeline would
        self.calls.append(kw)
        n = kw["num_images_per_prompt"]
        imgs = []
        for i in range(n):
            a = (np.arange(kw["height"] * kw["width"] * 3).reshape(kw["height"], kw["width"], 3) * (i + 3) +
                 int(draw[0] * 100)) % 256
            imgs.append(Image.fromarray(a.astype(np.uint8)))
        return SimpleNamespace(images=imgs)


class FakeSam:
    def generate(self, image):
        h, w = image.shape[:2]
        out = []
        for i, (y0, x0, dy, dx) in enumerate([(0, 0, h // 2, w // 2), (h // 4, w // 4, h // 2, w // 2), (h // 2, 0, h // 3, w)]):
            m = np.zeros((h, w), dtype=bool)
            m[y0:y0 + dy, x0:x0 + dx] = True
            out.append({"segmentation": m, "area": int(m.sum()) + (5 - i)})
        return out


def _inputs():
    g = np.random.RandomState(0)
    image = g.randint(0, 256, (90, 120, 3)).astype(np.uint8)
    mask = np.zeros((90, 120, 3), dtype=np.uint8)
    mask[20:60, 30:90] = 255
    src = {"image": image, "mask": mask}
    args = (src, False, None, 0.5, False, "a photo of a cat, best quality, extremely detailed", "lowres, bad anatomy, worst quality",
            2, 64, 64, 4, False, 9.0, 1234, 0.0)
    kwargs = dict(enable_tile=True, refine_alignment_ratio=0.95, refine_image_resolution=128, alpha_weight=0.0,
                  use_scale_map=False, condition_model="EditAnything")
    return args, kwargs


def _model(cls_or_obj, pipe, tile):
    m = object.__new__(cls_or_obj)
    m.device = torch.device("cpu")
    m.use_blip = False
    m.default_controlnet_path = app.config_dict["LAION Pretrained(v0-4)-SD15"]
    m.base_model_path, m.lora_model_path = "base", None
    m.defalut_enable_all_generate, m.extra_inpaint, m.last_ref_infer = False, True, False
    m.pipe, m.tile_pipe = pipe, tile
    m.sam_generator, m.mask_predictor = FakeSam(), None
    return m


def encode(v):
    """A recorded call / result as plain tensors, lists and dicts (what torch.load reads back without pickle)."""
    if torch.is_tensor(v):
        return v.as_subclass(torch.Tensor)       # input_ids and what derives from them are _Ids
    if isinstance(v, Image.Image):
        return {"__pil__": v.mode, "__data__": torch.from_numpy(np.array(v))}
    if isinstance(v, np.ndarray):
        return {"__ndarray__": torch.from_numpy(v)}
    if isinstance(v, torch.Generator):
        return {"__generator__": None}            # compared through the recorded generator_state
    if isinstance(v, dict):
        return {k: encode(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return [encode(x) for x in v]
    return v


def decode(v):
    if isinstance(v, dict) and "__pil__" in v:
        img = Image.fromarray(v["__data__"].numpy())
        return img if img.mode == v["__pil__"] else img.convert(v["__pil__"])
    if isinstance(v, dict) and "__ndarray__" in v:
        return v["__ndarray__"].numpy()
    if isinstance(v, dict) and "__generator__" in v:
        return torch.Generator()
    if isinstance(v, dict):
        return {k: decode(x) for k, x in v.items()}
    if isinstance(v, list):
        return [decode(x) for x in v]
    return v


def _same(a, b, path=""):
    if torch.is_tensor(a):
        assert torch.is_tensor(b) and a.dtype == b.dtype and a.shape == b.shape, (path, a.dtype, getattr(b, "dtype", None))
        assert torch.equal(a.cpu(), b.cpu()), path
    elif isinstance(a, Image.Image):
        assert isinstance(b, Image.Image) and a.size == b.size and a.mode == b.mode, path
        assert np.array_equal(np.array(a), np.array(b)), path
    elif isinstance(a, np.ndarray):
        assert np.array_equal(a, b), path
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _same(x, y, f"{path}[{i}]")
    elif isinstance(a, torch.Generator):
        pass
    else:
        assert a == b, (path, a, b)


def test_process_hands_the_pipelines_exactly_what_the_reference_does(monkeypatch):
    monkeypatch.setenv("EA_SAVE_INPUT", "0")
    args, kwargs = _inputs()
    ref = decode(torch.load(os.path.join(GOLD, "ref_app_process.pt")))     # the reference's process, np.random.seed(5)
    r_tile, r_res, r_masks, r_prompt = ref["result"]
    our_pipe, our_tile = SpyPipe(), SpyPipe()
    ours = _model(app.EditAnythingLoraModel, our_pipe, our_tile)
    np.random.seed(5)
    o_tile, o_res, o_masks, o_prompt = ours.process(*args, **kwargs)
    assert ref["n_main_calls"] == len(our_pipe.calls) == 1 and len(ref["calls"]) - 1 == len(our_tile.calls) == 2
    for rc, oc in zip(ref["calls"], our_pipe.calls + our_tile.calls):
        # the reference forwards the (unused, None-valued) reference-only keywords as well
        extra = {k: v for k, v in rc.items() if k not in oc}
        assert all(v is None or k.startswith(("attention_auto", "gn_auto", "style_fid", "reference_", "ref_")) for k, v in extra.items()), extra
        for k in oc:
            _same(rc[k], oc[k], k)
    _same(r_tile, o_tile, "results_tile")
    _same(r_res, o_res, "results")
    _same(r_masks, o_masks, "[full_segmask, mask]")
    assert r_prompt == o_prompt
    main = our_pipe.calls[0]
    assert main["controlnet_conditioning_image"][0].dtype == torch.float16
    assert float(main["controlnet_conditioning_image"][0].max()) > 1.5          # the id map is NOT normalised
    assert float(main["controlnet_conditioning_image"][1].min()) == -1.0         # masked pixels of the inpaint condition
    assert main["controlnet_conditioning_scale"] == [0.5, 1.0] and main["height"] == 64 and main["width"] == 64
    assert our_tile.calls[0]["alignment_ratio"] == 0.95 and our_tile.calls[0]["controlnet_conditioning_scale"] == 1.0


def test_process_end_to_end_on_tiny_engines_from_input_data_pkl(tmp_path, monkeypatch):
    from editanything_b200.denoise import DenoiseEngine
    from editanything_b200.pipeline import StableDiffusionControlNetInpaintPipeline
    from editanything_b200.schedulers import UniPCMultistepScheduler
    from editanything_b200.unet_spec import TINY, make_state_dict
    from editanything_b200.vae import VaeEngine, make_vae_state_dict
    from editanything_b200.vae_spec import VaeConfig
    from tests import cpu_ops
    monkeypatch.chdir(tmp_path)
    dev = torch.device("cpu")
    vcfg = VaeConfig(ch=64, ch_mult=(1, 1, 1, 1), num_res_blocks=1)
    vsd = dict(make_vae_state_dict(vcfg, 61, part="encoder"))
    vsd.update(make_vae_state_dict(vcfg, 62))
    vae = VaeEngine(vcfg, vsd, dev, backend=cpu_ops)
    usd = make_state_dict(TINY, "unet", 51)
    main_eng = DenoiseEngine(TINY, usd, [make_state_dict(TINY, "controlnet", 52), make_state_dict(TINY, "controlnet", 53)], dev, backend=cpu_ops)
    tile_eng = DenoiseEngine(TINY, None, [make_state_dict(TINY, "controlnet", 54)], dev, backend=cpu_ops, unet_packed=main_eng.unet)
    assert tile_eng.unet is main_eng.unet                                      # the tile pass shares the UNet weights
    tok, enc = _Tok(), _Enc(TINY.context_dim)

    def mk(eng):
        p = StableDiffusionControlNetInpaintPipeline(eng, vae=vae, text_encoder=enc, tokenizer=tok)
        p.scheduler = UniPCMultistepScheduler.from_config(p.scheduler.config)   # editany_lora.py:383,418
        return p
    model = app.EditAnythingLoraModel(base_model_path="base", lora_model_path=None, use_blip=False, sam_generator=FakeSam(),
                                      mask_predictor=object(), tile_model=mk(tile_eng), pipe=mk(main_eng))
    args, kwargs = _inputs()
    args = args[:10] + (20,) + args[11:]      # 20 steps: with 4, alignment_ratio 0.95 covers the last step and the
    #                                           reference's timesteps[i + 1] (:1652) raises IndexError - here too
    with open("input_data.pkl", "wb") as f:                                     # what @save_input_to_file writes
        pickle.dump({"args": args, "kwargs": kwargs}, f)
    data = pickle.load(open("input_data.pkl", "rb"))
    refined, output, ref, text = model.process(*data["args"], **data["kwargs"])  # editany_nogradio.py:15
    assert text == args[5] and len(output) == 2 and len(refined) == 2
    assert all(isinstance(i, Image.Image) and i.size == (64, 64) for i in output)
    assert all(isinstance(i, Image.Image) and i.size == (128, 128) for i in refined)
    assert isinstance(ref[0], Image.Image) and isinstance(ref[1], Image.Image) and ref[1].size == (64, 64)
    assert os.path.exists("input_data.pkl")                                     # re-written by the decorator
    again = model.process(*data["args"], **data["kwargs"])
    assert all(np.array_equal(np.array(a), np.array(b)) for a, b in zip(output + refined, again[1] + again[0]))   # seeded
    with pytest.raises(NotImplementedError):
        model.process(*data["args"], **{**data["kwargs"], "ref_image": {"image": None, "mask": None}})


def test_engines_survive_inference_mode_callers():
    """`process` runs under @torch.inference_mode() like the reference (editany_lora.py:609); engine buffers created
    during such a call must stay usable from a later call outside inference mode (in-place updates)."""
    from editanything_b200.denoise import DenoiseEngine
    from editanything_b200.unet_spec import TINY, make_state_dict
    from oracle.inputs import make_inputs
    from tests import cpu_ops
    eng = DenoiseEngine(TINY, make_state_dict(TINY, "unet", 1), [make_state_dict(TINY, "controlnet", 2)], torch.device("cpu"),
                        backend=cpu_ops)
    x, ctx, hints = make_inputs(TINY, 2, 8, 7, 1, n_controlnets=1)
    with torch.inference_mode():
        eng.prepare(ctx, hints, [1.0])
        eng.begin(x[:1], 5.0, use_graph=False)
        eng.step(501, 0.3, 0.4)
    eng.prepare(ctx, hints, [1.0])                 # outside: copies into the buffers created above
    eng.begin(x[:1], 5.0, use_graph=False)
    eng.step(481, 0.32, 0.42)
    assert not eng.lat.is_inference() and torch.isfinite(eng.latents()).all()
