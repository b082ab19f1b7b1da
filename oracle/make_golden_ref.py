"""Generate the tests/golden/ref_*.pt fixtures by running the reference's own code (needs the reference tree,
see oracle/ref_shim.py).

    python -m oracle.make_golden_ref

Each fixture holds what a CPU test used to obtain by importing the reference at test time, for the test's own
inputs, so that the comparison runs on any machine:
  ref_unet_modules.pt  cldm ControlNet / ControlledUnetModel outputs (tests/test_oracle.py)
  ref_vae_modules.pt   ldm Decoder / Encoder outputs (tests/test_vae_cpu.py)
  ref_host.pt          annotator/util.py helpers and editany_lora.py host functions (tests/test_host_semantics_cpu.py)
  ref_app_process.pt   EditAnythingLoraModel.process: every pipeline call and the result (tests/test_app_cpu.py)
Large outputs are stored as a fixed sample (`sample`) or, where the test asks for bit equality, as a digest."""
import ast
import os
import random
import sys

import numpy as np
import torch
from PIL import Image

from oracle import ref_shim

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def sample(t, k=256, seed=0):
    """A fixed, seeded sample of `t`'s elements: flat indices, values and the largest magnitude of the whole tensor."""
    flat = t.detach().reshape(-1).float()
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:k].sort().values
    return {"idx": idx.to(torch.int32), "val": flat[idx].clone(), "absmax": float(flat.abs().max())}


def unet_modules():
    """tests/test_oracle.py::test_oracle_matches_live_reference_modules, per config."""
    from editanything_b200.unet_spec import TINY, TINY21, make_state_dict
    from oracle.inputs import make_inputs
    out = {}
    for name, cfg in (("tiny_sd15", TINY), ("tiny_sd21", TINY21)):
        usd = make_state_dict(cfg, "unet", 1)
        csd = make_state_dict(cfg, "controlnet", 2)
        unet, cns = ref_shim.build_reference_nets(cfg, usd, [csd])
        x, ctx, hints = make_inputs(cfg, 2, 16, 9, 3, n_controlnets=1)
        ref, control = ref_shim.reference_apply_model(unet, cns, x, torch.tensor([321, 321]), ctx, hints, [0.7])
        out[name] = {"eps": ref.clone(), "control": [sample(c, seed=i) for i, c in enumerate(control)]}
    torch.save(out, os.path.join(GOLD, "ref_unet_modules.pt"))


def vae_modules():
    """tests/test_vae_cpu.py: test_oracle_matches_reference_decoder / test_encode_oracle_matches_reference_encoder."""
    from editanything_b200.vae_spec import VAE_TINY, make_vae_state_dict
    from oracle import vae_oracle as V
    from oracle.make_golden_vae import make_image, make_latents
    cfg = VAE_TINY
    z = make_latents(cfg, 2, 12, 5) / cfg.scaling_factor
    dec = V.reference_decoder(cfg, make_vae_state_dict(cfg, 21))(z)
    enc = V.reference_encoder(cfg, make_vae_state_dict(cfg, 31, part="encoder"))(make_image(2, 24, 6))
    torch.save({"decoded": dec.clone(), "moments": enc.clone()}, os.path.join(GOLD, "ref_vae_modules.pt"))


def _ref_source_functions(ns, *names):
    """Compile exactly the named top-level functions of the reference's editany_lora.py (its module-level imports -
    diffusers, gradio, segment_anything - are not needed by them) into `ns`."""
    tree = ast.parse(open(os.path.join(ref_shim.REFERENCE_ROOT, "editany_lora.py")).read())
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            exec(compile(ast.Module([node], []), "editany_lora.py", "exec"), ns)
    return [ns[n] for n in names]


def _ref_util():
    if ref_shim.REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, ref_shim.REFERENCE_ROOT)
    import annotator.util as U
    return U


def host():
    """tests/test_host_semantics_cpu.py, test by test, with the same inputs."""
    from tests.test_host_semantics_cpu import _Enc, _Tok, _anns, digest, long_prompt
    from types import SimpleNamespace
    ref_show, ref_mic, ref_gpe = _ref_source_functions({"np": np, "Image": Image, "torch": torch}, "show_anns",
                                                       "make_inpaint_condition", "get_pipeline_embeds")
    out = {}
    np.random.seed(11)
    img, res = ref_show(_anns(3))
    empty_is_none = ref_show([]) is None
    many = [{"segmentation": np.eye(300, dtype=bool)[i:i + 1].repeat(2, 0), "area": 2} for i in range(300)]
    np.random.seed(1)
    many_res = ref_show(many)[1]
    out["show_anns"] = {"image": torch.from_numpy(np.array(img)), "res": torch.from_numpy(res),
                        "empty_is_none": empty_is_none, "many_res": torch.from_numpy(many_res)}
    g = np.random.RandomState(5)
    img = g.randint(0, 256, (32, 48, 3)).astype(np.uint8)
    mask = np.zeros((32, 48, 3), dtype=np.uint8)
    mask[8:20, 10:30] = 255
    out["make_inpaint_condition"] = ref_mic(img.copy(), mask)
    U = _ref_util()
    g = np.random.RandomState(7)
    out["HWC3"] = [digest(U.HWC3(g.randint(0, 256, shape).astype(np.uint8)))
                   for shape in [(50, 70), (50, 70, 1), (50, 70, 3), (50, 70, 4)]]
    img = g.randint(0, 256, (300, 421, 3)).astype(np.uint8)
    out["resize_image"] = {res: digest(U.resize_image(img, res)) for res in (128, 512, 1024)}
    out["resize_points"] = [list(p) for p in U.resize_points([(10, 20, 1), (333, 7, 0)], img.shape, 512)]
    m = np.zeros((40, 60, 3), dtype=np.uint8)
    m[5:9, 11:30] = 1
    out["get_bounding_box"] = [int(v) for v in U.get_bounding_box(m)]
    pipe = SimpleNamespace(tokenizer=_Tok(), text_encoder=_Enc())
    out["get_pipeline_embeds"] = [tuple(t.clone() for t in ref_gpe(pipe, p, n, "cpu"))
                                  for p, n in [(long_prompt, "lowres, bad anatomy"), ("short", long_prompt), ("a cat", "a dog")]]
    torch.save(out, os.path.join(GOLD, "ref_host.pt"))


def _reference_model_class():
    """The reference's EditAnythingLoraModel with ONLY `process`, `get_sam_control` (their unmodified source) and
    the module-level helpers they call, compiled in a namespace of stand-ins for the absent third-party imports."""
    import cv2
    import einops
    from editanything_b200 import host as H
    U = _ref_util()
    ns = {"np": np, "torch": torch, "cv2": cv2, "einops": einops, "random": random, "Image": Image, "PIL": __import__("PIL"),
          "os": os, "HWC3": U.HWC3, "resize_image": U.resize_image, "get_bounding_box": U.get_bounding_box,
          "seed_everything": H.seed_everything, "StableDiffusionControlNetInpaintMixingPipeline": type("Mix", (), {}),
          "prepare_mask_image": None, "obtain_generation_model": None}
    __import__("PIL.Image")
    _ref_source_functions(ns, "show_anns", "make_inpaint_condition", "get_pipeline_embeds")
    tree = ast.parse(open(os.path.join(ref_shim.REFERENCE_ROOT, "editany_lora.py")).read())
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name == "EditAnythingLoraModel":
            keep = [n for n in node.body if isinstance(n, ast.FunctionDef) and n.name in ("process", "get_sam_control")]
            for n in keep:
                n.decorator_list = []          # @torch.inference_mode() / @save_input_to_file: not part of the arithmetic
            node.body = keep
            exec(compile(ast.Module([node], []), "editany_lora.py", "exec"), ns)
    return ns["EditAnythingLoraModel"]


def app_process():
    """tests/test_app_cpu.py::test_process_hands_the_pipelines_exactly_what_the_reference_does: the reference's
    `process` on the test's inputs with the test's spy pipelines."""
    from tests.test_app_cpu import SpyPipe, _inputs, _model, encode
    torch.Tensor.cuda = lambda self, *a, **k: self              # the reference hard-codes .cuda()
    args, kwargs = _inputs()
    pipe, tile = SpyPipe(), SpyPipe()
    model = _model(_reference_model_class(), pipe, tile)
    np.random.seed(5)
    result = model.process(*args, **kwargs)
    torch.save(encode({"calls": pipe.calls + tile.calls, "n_main_calls": len(pipe.calls), "result": list(result)}),
               os.path.join(GOLD, "ref_app_process.pt"))


if __name__ == "__main__":
    if not ref_shim.available():
        sys.exit("reference tree not present: set EA_REFERENCE_ROOT")
    os.environ["EA_SAVE_INPUT"] = "0"
    torch.manual_seed(0)
    unet_modules()
    vae_modules()
    host()
    app_process()
    for f in sorted(os.listdir(GOLD)):
        if f.startswith("ref_"):
            print(f, os.path.getsize(os.path.join(GOLD, f)), "bytes")
