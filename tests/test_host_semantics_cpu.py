"""Host semantics of SURVEY.md §8a rows R2 / R3 / R4 (`editanything_b200.host`) against the REFERENCE's own
functions: annotator/util.py and the show_anns / make_inpaint_condition / get_pipeline_embeds definitions of
editany_lora.py, run unmodified on these tests' inputs by oracle/make_golden_ref.py.  Their results are stored in
tests/golden/ref_host.pt (bit-exact comparisons of large arrays as a digest)."""
import functools
import hashlib
import os
from types import SimpleNamespace

import numpy as np
import torch

from editanything_b200 import host

GOLD_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_host.pt")


@functools.lru_cache(maxsize=None)
def _gold():
    return torch.load(GOLD_PATH)


def digest(a):
    """dtype, shape and SHA-256 of an array's bytes: equal digests <=> np.array_equal with the same dtype."""
    a = np.ascontiguousarray(a)
    return f"{a.dtype}{a.shape}:{hashlib.sha256(a.tobytes()).hexdigest()}"


def _anns(seed, n=7, H=48, W=64):
    g = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        m = np.zeros((H, W), dtype=bool)
        y0, x0 = g.randint(0, H - 8), g.randint(0, W - 8)
        m[y0:y0 + g.randint(4, 30), x0:x0 + g.randint(4, 40)] = True
        out.append({"segmentation": m, "area": int(m.sum())})
    return out


def test_show_anns_matches_reference_including_the_ordering_quirk():
    ref = _gold()["show_anns"]
    anns = _anns(3)
    img_r, res_r = ref["image"].numpy(), ref["res"].numpy()          # after np.random.seed(11)
    np.random.seed(11)
    img_o, res_o = host.show_anns(anns)
    assert res_o.dtype == res_r.dtype == np.float64
    assert np.array_equal(res_o, res_r)
    assert np.array_equal(np.array(img_o), img_r)
    # the quirk: ids follow the generator's order, not the area order - sorting the input changes the map
    srt = sorted(anns, key=lambda a: a["area"], reverse=True)
    np.random.seed(11)
    assert not np.array_equal(host.show_anns(srt)[1], res_o)
    assert host.show_anns([]) is None and ref["empty_is_none"]
    # more than 255 masks: the id spills into channel 1
    many = [{"segmentation": np.eye(300, dtype=bool)[i:i + 1].repeat(2, 0), "area": 2} for i in range(300)]
    np.random.seed(1)
    r_o = host.show_anns(many)[1]
    assert np.array_equal(r_o, ref["many_res"].numpy()) and r_o[:, :, 1].max() == 1


def test_make_inpaint_condition_matches_reference():
    g = np.random.RandomState(5)
    img = g.randint(0, 256, (32, 48, 3)).astype(np.uint8)
    mask = np.zeros((32, 48, 3), dtype=np.uint8)
    mask[8:20, 10:30] = 255
    a = host.make_inpaint_condition(img.copy(), mask)
    b = _gold()["make_inpaint_condition"]
    assert a.dtype == b.dtype and a.shape == b.shape == (1, 3, 32, 48)
    assert torch.equal(a, b)
    assert float(a.min()) == -1.0


def test_image_helpers_match_annotator_util():
    g = np.random.RandomState(7)
    for shape, ref in zip([(50, 70), (50, 70, 1), (50, 70, 3), (50, 70, 4)], _gold()["HWC3"]):
        x = g.randint(0, 256, shape).astype(np.uint8)
        assert digest(host.HWC3(x)) == ref
    img = g.randint(0, 256, (300, 421, 3)).astype(np.uint8)
    for res in (128, 512, 1024):
        a = host.resize_image(img, res)
        assert a.shape[0] % 64 == 0 and a.shape[1] % 64 == 0
        assert digest(a) == _gold()["resize_image"][res], res
    pts = [(10, 20, 1), (333, 7, 0)]
    assert [list(p) for p in host.resize_points(pts, img.shape, 512)] == _gold()["resize_points"]
    m = np.zeros((40, 60, 3), dtype=np.uint8)
    m[5:9, 11:30] = 1
    assert [int(v) for v in host.get_bounding_box(m)] == _gold()["get_bounding_box"] == [11, 5, 29, 8]


class _Tok:
    """Word-level tokenizer with the call surface get_pipeline_embeds uses (CLIPTokenizer-like: BOS ... EOS, pad)."""
    model_max_length = 8

    def __call__(self, text, return_tensors="pt", truncation=False, padding=None, max_length=None):
        ids = [1] + [3 + (sum(map(ord, w)) % 50) for w in text.replace(",", " ").split()] + [2]
        if padding == "max_length" and max_length is not None:
            ids = ids + [0] * (max_length - len(ids))
        return SimpleNamespace(input_ids=torch.tensor([ids]))


class _Enc(torch.nn.Module):
    def __init__(self):
        super().__init__()
        torch.manual_seed(0)
        self.emb = torch.nn.Embedding(64, 16)

    def forward(self, ids):
        x = self.emb(ids)
        return (x + x.cumsum(1) * 0.1,)          # depends on the position inside the window


long_prompt = "a photo of a very long prompt with many many words, best quality, extremely detailed, more words here"


def test_get_pipeline_embeds_windows_match_reference():
    pipe = SimpleNamespace(tokenizer=_Tok(), text_encoder=_Enc())
    cases = [(long_prompt, "lowres, bad anatomy"), ("short", long_prompt), ("a cat", "a dog")]
    for (p, n), b in zip(cases, _gold()["get_pipeline_embeds"]):
        a = host.get_pipeline_embeds(pipe, p, n, "cpu")
        assert a[0].shape == a[1].shape == b[0].shape
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert host.get_pipeline_embeds(pipe, long_prompt, "x", "cpu")[0].shape[1] > _Tok.model_max_length


def test_seed_everything_seeds_all_generators():
    import random
    host.seed_everything(123)
    a = (random.random(), np.random.rand(), torch.rand(1).item())
    host.seed_everything(123)
    assert a == (random.random(), np.random.rand(), torch.rand(1).item())
    assert os.environ["PL_GLOBAL_SEED"] == "123"
