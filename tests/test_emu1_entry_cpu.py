"""CPU: the Emu1 example entry points (emu_b200/emu1/inference.py, utils.py, image_inference.py — BASELINE configs[0] is the
captioning call of the reference's inference.py) — input preparation bit-identical to the reference's own `utils.process_img`,
frame selection, prompt assembly and the generate calls the helpers make."""
import os
import types

import numpy as np
import torch
from PIL import Image


def _picture(seed, size=(93, 61)):
    rng = np.random.RandomState(seed)
    return Image.fromarray(rng.randint(0, 256, (size[1], size[0], 3), dtype=np.uint8))


def test_process_img_formula():
    """Pillow default-filter resize to 224 x 224 on uint8, (x / 255 - mean) / std in float64, one rounding to fp32, CHW"""
    from emu_b200.emu1.utils import process_img
    from emu_b200.emu2.constants import OPENAI_DATASET_MEAN, OPENAI_DATASET_STD
    img = _picture(0)
    x = process_img(img=img, device=torch.device("cpu"))
    assert x.shape == (1, 3, 224, 224) and x.dtype == torch.float32
    ref = (np.array(img.resize((224, 224))) / 255. - OPENAI_DATASET_MEAN) / OPENAI_DATASET_STD
    assert torch.equal(x[0], torch.tensor(ref).to(torch.float).permute(2, 0, 1))


def test_process_img_and_get_index_vs_live_reference():
    """process_img bitwise and get_index exactly as the reference's Emu1/utils.py returned them
    (tests/golden/gen_golden_reference_checks.py)"""
    from helpers import assert_equal_digest
    from emu_b200.emu1 import utils as mine
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.pt"))["emu1_utils"]
    pictures = ((1, (640, 480)), (2, (100, 333)), (3, (224, 224)))
    assert len(gold["process_img"]) == len(pictures)
    for (seed, size), want in zip(pictures, gold["process_img"]):
        assert_equal_digest(mine.process_img(img=_picture(seed, size), device=torch.device("cpu")), want)
    frame_cases = ((300, 8), (9, 8), (17, 4), (1000, 8))
    assert len(gold["get_index"]) == len(frame_cases)
    for (frames, segs), want in zip(frame_cases, gold["get_index"]):
        assert np.array_equal(mine.get_index(frames, segs), want.numpy())


class _FakeEmu:
    def __init__(self):
        self.calls = []

    def generate(self, samples, **kw):
        self.calls.append((samples, kw))
        return ["  an answer  "]


def test_inference_helpers_build_the_reference_prompts(monkeypatch):
    from emu_b200.emu1 import inference as I
    fake = _FakeEmu()
    monkeypatch.setattr(I, "emu_model", fake)
    monkeypatch.setattr(I, "args", types.SimpleNamespace(device=torch.device("cpu")))
    ph = "[IMG]" + "<image>" * 32 + "[/IMG]"
    assert I.image_placeholder == ph
    a, b = torch.zeros(1, 3, 4, 4), torch.ones(1, 3, 4, 4)
    images, text = I.interleave([a, "There are two dogs.", b, "There are three pandas.", a])
    assert len(images) == 3 and text == ph + "There are two dogs." + ph + "There are three pandas." + ph
    assert I.Emu_inference(images, text, instruct=False) == "an answer"
    samples, kw = fake.calls[-1]
    assert samples["prompt"] == text and samples["image"].shape == (3, 3, 4, 4)
    assert kw == dict(max_new_tokens=128, num_beams=5, length_penalty=0.0, repetition_penalty=1.0)
    I.Emu_inference([a], ph + "what is the man doing?", system=I.image_system_msg)
    assert fake.calls[-1][0]["prompt"] == I.image_system_msg + " [USER]: " + ph + "what is the man doing? [ASSISTANT]:"
    I.Emu_inference([a], "hi", system="")                    # an empty system message: the leading blank is stripped
    assert fake.calls[-1][0]["prompt"] == "[USER]: hi [ASSISTANT]:"
    I.Emu_instruct_caption(a)
    samples, kw = fake.calls[-1]
    assert samples["prompt"] == (I.image_system_msg + " [USER]: " + ph + "Please provide an accurate and concise description of "
                                 "the given image. [ASSISTANT]: The image depicts a photo of")
    assert kw == dict(max_new_tokens=512, num_beams=5, length_penalty=0.0, repetition_penalty=1.0)
    assert I.parse_args(["--instruct", "--ckpt-path", "x.pt"]).instruct is True and I.parse_args([]).ckpt_path == ""


def test_image_inference_cases(tmp_path, monkeypatch):
    from emu_b200.emu1 import image_inference as G
    seen = []

    class Pipe:
        def __call__(self, inputs, height, width, guidance_scale):
            seen.append(([type(i).__name__ for i in inputs], height, width, guidance_scale))
            return Image.new("RGB", (8, 8)), (True if guidance_scale == 10.0 else None)
    monkeypatch.setattr(G.Image, "open", lambda path: Image.new("RGB", (5, 5)))
    monkeypatch.chdir(tmp_path)
    for case in G.CASES:
        G.run_case(Pipe(), *case)
    assert [s[1:] for s in seen] == [(512, 512, 7.5), (512, 512, 7.5), (512, 512, 10.0)]
    assert seen[0][0] == ["Image", "Image"] and seen[1][0] == ["str"] and seen[2][0] == ["str", "Image", "str", "Image", "str"]
    names = sorted(p.name for p in tmp_path.iterdir())
    assert names == ["image_blend_result.jpg", "text2image_result.jpg"]      # the flagged third image is not written
