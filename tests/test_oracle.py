"""CPU suite: the oracle restatement against (a) the reference-generated golden vectors and
(b) the outputs of the reference's own modules, recorded by oracle/make_golden_ref.py."""
import os

import numpy as np
import pytest
import torch

from editanything_b200.denoise import ddim_schedule
from editanything_b200.unet_spec import SD15, SD21, TINY, TINY21, build_topology, make_state_dict, param_shapes
from oracle import unet_oracle as O
from oracle.inputs import make_inputs

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CFGS = {"tiny_sd15": TINY, "tiny_sd21": TINY21, "tiny_sd15_32": TINY}


def _oracle_eps(cfg, m, t):
    usd = make_state_dict(cfg, "unet", m["unet_seed"])
    csds = [make_state_dict(cfg, "controlnet", s) for s in m["cn_seeds"]]
    x, ctx, hints = make_inputs(cfg, m["B"], m["lat"], m["L"], m["in_seed"], n_controlnets=len(csds))
    ut, ct = build_topology(cfg), build_topology(cfg, with_decoder=False)
    with torch.no_grad():
        return O.apply_model(usd, ut, [(sd, ct) for sd in csds], x, torch.full((m["B"],), t), ctx, hints, m["scales"])


@pytest.mark.parametrize("name", list(CFGS))
def test_oracle_reproduces_reference_golden(name):
    g = torch.load(os.path.join(GOLD, name + ".pt"))
    m = g["meta"]
    for t in m["timesteps"]:
        eps = _oracle_eps(CFGS[name], m, t)
        assert (eps - g[f"eps_t{t}"]).abs().max().item() < 5e-5


def test_param_counts_match_published_sizes():
    # SURVEY.md §6: UNet 859.5 M; ControlNet 361.3 M (SD1.5), 865.9 M / 364.2 M (SD2.1)
    def count(cfg, kind):
        return sum(int(np.prod(s)) for s, _ in param_shapes(cfg, kind).values())
    assert count(SD15, "unet") == 859520964
    assert count(SD15, "controlnet") == 361279120
    assert abs(count(SD21, "unet") - 865.9e6) < 0.1e6
    assert abs(count(SD21, "controlnet") - 364.2e6) < 0.1e6


def test_ddim_schedule_matches_reference_tables():
    g = torch.load(os.path.join(GOLD, "ddim.pt"))
    for S in (20, 30, 50):
        ts, a, ap = ddim_schedule(S)
        ref = g[f"S{S}"]
        assert list(ts[::-1]) == ref["timesteps"].tolist()
        assert np.allclose(a[::-1], ref["alphas"].numpy(), rtol=1e-12)
        assert np.allclose(ap[::-1], ref["alphas_prev"].numpy(), rtol=1e-12)
        assert float(ref["sigmas"].abs().max()) == 0.0
        ots, oa, oap = O.make_ddim_schedule(S)
        assert list(ots) == ref["timesteps"].tolist() and np.allclose(oa, ref["alphas"].numpy(), rtol=1e-6)
    assert len(ddim_schedule(30)[0]) == 31   # reference quirk: S=30 -> 31 steps (util.py:48-49)


def test_ddim_step_matches_reference_p_sample():
    g = torch.load(os.path.join(GOLD, "ddim.pt"))["p_sample"]
    ts, a, ap = O.make_ddim_schedule(50)
    i = g["index"]
    x_prev, x0 = O.ddim_step(g["x"], g["e_uncond"], g["e_cond"], g["guidance"], float(a[i]), float(ap[i]))
    assert (x_prev - g["x_prev"]).abs().max().item() < 1e-5
    assert (x0 - g["pred_x0"]).abs().max().item() < 1e-4


@pytest.mark.parametrize("cfg", [TINY, TINY21])
def test_oracle_matches_live_reference_modules(cfg):
    """The reference's ControlNet + ControlledUnetModel, loaded strictly with these state dicts (so the topology is
    restated right), gave `eps` and the scaled control residuals (a fixed sample of each) in ref_unet_modules.pt."""
    g = torch.load(os.path.join(GOLD, "ref_unet_modules.pt"))["tiny_sd15" if cfg == TINY else "tiny_sd21"]
    usd = make_state_dict(cfg, "unet", 1)
    csd = make_state_dict(cfg, "controlnet", 2)
    x, ctx, hints = make_inputs(cfg, 2, 16, 9, 3, n_controlnets=1)
    t = torch.tensor([321, 321])
    ut, ct = build_topology(cfg), build_topology(cfg, with_decoder=False)
    with torch.no_grad():
        outs = O.controlnet_forward(csd, ct, x, hints[0], t, ctx)
        eps = O.apply_model(usd, ut, [(csd, ct)], x, t, ctx, hints, [0.7])
    assert len(outs) == len(g["control"]) == 13
    for a_, b_ in zip(outs, g["control"]):
        assert (0.7 * a_.reshape(-1)[b_["idx"].long()] - b_["val"]).abs().max().item() < 2e-5 * max(1.0, b_["absmax"])
    assert (eps - g["eps"]).abs().max().item() < 5e-5
