"""CPU: host-side logic that mirrors the reference without touching the GPU — prompt assembly of the chat
pipeline, the Euler scheduler tables against the oracle restatement, config translation."""
import json
import os

import torch

from oracle import diffusion_oracle as D

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# the reference's published Emu2-Gen configuration files (tests/golden/gen_golden_reference_checks.py copies them)
REF_DIFFUSION_CONFIG = os.path.join(GOLDEN, "emu2_diffusion_config")


def test_euler_tables_match_oracle():
    from emu_b200.emu2.scheduler import EulerDiscreteScheduler
    s = EulerDiscreteScheduler()
    for n in (50, 20, 7):
        s.set_timesteps(n)
        ts, sig, init = D.euler_tables(n)
        assert torch.equal(s.timesteps, ts)
        assert torch.allclose(s.sigmas, sig, rtol=0, atol=0)
        assert abs(s.init_noise_sigma - init) < 1e-6
    s.set_timesteps(50)
    assert s.timesteps[0] == 981 and s.timesteps[-1] == 1 and s.sigmas[-1] == 0
    # external anchor (diffusers is not installable here, SURVEY §8c): the scaled-linear 0.00085 -> 0.012 / 1000-step noise
    # schedule of Emu2/emu/conf/diffusion_config/scheduler/scheduler_config.json has the published Stable-Diffusion sigma
    # range sigma_min = 0.0292, sigma_max = 14.6146 (k-diffusion / SD v1 sampling configs quote exactly these)
    assert abs(float(s._sigmas_all[-1]) - 14.6146) < 1e-3
    assert abs(float(s._sigmas_all[0]) - 0.0292) < 1e-4


class _FakeModel:
    def __init__(self):
        self.calls = []

    def device(self):
        return torch.device("cpu")

    def dtype(self):
        return torch.float32

    def generate(self, **kw):
        self.calls.append(kw)
        return ["ok"]


def test_chat_prompt_assembly():
    from PIL import Image
    from emu_b200.emu2.chat import EmuChatGeneration
    from emu_b200.emu2 import constants as K
    fm = _FakeModel()
    pipe = EmuChatGeneration(fm)
    img = Image.new("RGB", (64, 48), (10, 200, 30))
    assert pipe.forward([img, "describe"], max_new_tokens=3) == "ok"
    kw = fm.calls[-1]
    assert kw["text"] == [K.DEFAULT_IMG_PLACEHOLDER + "describe"] and kw["image"].shape == (1, 3, 448, 448)
    assert kw["num_beams"] == 5 and kw["length_penalty"] == -1          # reference defaults
    pipe.forward([[img, "what is this?"], ["a cat"], ["and this?", img]], is_grounding=True)
    t = fm.calls[-1]["text"][0]
    assert t.startswith(K.GROUND_SYSTEM_MESSAGE + " [USER]: " + K.DEFAULT_IMG_PLACEHOLDER + "what is this?")
    assert " [ASSISTANT]: a cat</s>[USER]: and this?" in t and t.endswith(" [ASSISTANT]:" + K.GRD_SYMBOL)
    assert fm.calls[-1]["image"].shape[0] == 2


def test_image_transform_matches_reference_formula():
    """Resize(448, bicubic) -> ToTensor -> Normalize(OPENAI mean/std)  (Emu2/emu/chat.py:35-39)."""
    from PIL import Image
    import numpy as np
    from emu_b200.emu2.diffusion import image_transform
    from emu_b200.emu2.constants import OPENAI_DATASET_MEAN, OPENAI_DATASET_STD
    rng = np.random.RandomState(0)
    img = Image.fromarray(rng.randint(0, 255, (40, 60, 3), dtype=np.uint8))
    x = image_transform(img)
    ref = np.asarray(img.resize((448, 448), resample=Image.BICUBIC), dtype=np.float32) / 255.0
    ref = (ref - np.array(OPENAI_DATASET_MEAN, dtype=np.float32)) / np.array(OPENAI_DATASET_STD, dtype=np.float32)
    assert x.shape == (3, 448, 448)
    assert np.allclose(x.permute(1, 2, 0).numpy(), ref, atol=1e-6)


def test_unet_config_translation_and_param_count():
    from emu_b200.emu2.diffusion import unet_config_from_json
    cfg = json.load(open(os.path.join(REF_DIFFUSION_CONFIG, "unet", "config.json")))
    u = unet_config_from_json(cfg)
    assert list(u.block_out_channels)[:3] == [320, 640, 1280] and list(u.transformer_layers)[:3] == [0, 2, 10]
    assert u.head_dim == 64 and u.cross_attention_dim == 1792 and u.projection_class_embeddings_input_dim == 3328
    n = sum(torch.Size(s).numel() for s in D.unet_param_shapes(D.EMU2_UNET).values())
    assert abs(n / 1e9 - 2.526) < 2e-3   # SURVEY.md §8a row a14: 2.526 B parameters from the reference's config
    import bench
    assert sum(torch.Size(s).numel() for _, s in bench.unet_param_shapes(bench.emu2_unet_json())) == n


def test_chat_prompt_assembly_vs_live_reference():
    """Prompt strings and image tensors of EmuChatGeneration._prepare_inputs / _prepare_chat_inputs are identical to what
    the UNMODIFIED reference (Emu2/emu/chat.py:121-195) returned (tests/golden/gen_golden_reference_checks.py), for
    plain, interleaved, video and multi-turn (grounding) inputs; image tensors bitwise, through their SHA-256."""
    from helpers import assert_equal_digest, chat_prompt_cases
    from emu_b200.emu2.chat import EmuChatGeneration
    gold = torch.load(os.path.join(GOLDEN, "reference_checks.pt"))["chat"]
    mine = EmuChatGeneration(_FakeModel())
    plain, chats = chat_prompt_cases()

    def same(x, d):
        assert (x is None) == (d is None)
        if x is not None:
            assert_equal_digest(x, d)
    assert len(plain) == len(gold["plain"]) and len(chats) == len(gold["chat"])
    for inp, b in zip(plain, gold["plain"]):
        a = mine._prepare_inputs(inp)
        assert a[0] == b["text"] and a[3:] == b["rest"]
        same(a[1], b["image"])
        same(a[2], b["video"])
    for (inp, grounding), b in zip(chats, gold["chat"]):
        a = mine._prepare_chat_inputs(inp, is_grounding=grounding)
        assert a[0] == b["text"]
        same(a[1], b["image"])


class _FakeEncoder:
    """records what EmuVisualGeneration asks of its multimodal encoder (Emu2/emu/diffusion.py:168-212)"""

    def __init__(self):
        self.calls = []

    def encode_image(self, image):
        self.calls.append(("encode_image", tuple(image.shape), float(image.abs().sum())))
        return torch.full((image.shape[0], 2, 3), 1.0 if float(image.abs().sum()) else -1.0)

    def generate_image(self, text, image=None):
        self.calls.append(("generate_image", list(text), None if image is None else tuple(image.shape)))
        return torch.full((len(text), 2, 3), 2.0 if text[0] else -2.0)


def _bare_visual_generation():
    from emu_b200.emu2.diffusion import EmuVisualGeneration
    g = EmuVisualGeneration.__new__(EmuVisualGeneration)   # host logic only: no engine behind it
    g.multimodal_encoder, g.negative_prompt, g.device_ = _FakeEncoder(), {}, torch.device("cpu")
    g.transform = lambda img, device=None: torch.ones(3, 4, 4) * img
    return g


def test_visual_generation_prompt_modes():
    """The two modes of the reference's _prepare_and_encode_inputs: pictures only -> autoencoding (encode_image, negative =
    the zero image, cached under "[NULL_IMAGE]"); anything with text -> generate_image on the concatenated text with one
    placeholder per picture (negative = the empty prompt, cached under ""); [cond; uncond] order; no CFG -> cond only."""
    g = _bare_visual_generation()
    enc = g.multimodal_encoder
    out = g._prepare_and_encode_inputs([5.0], True)           # a "picture" (the fake transform scales a ones tensor)
    assert out.shape[0] == 2 and float(out[0, 0, 0]) == 1.0 and float(out[1, 0, 0]) == -1.0
    assert [c[0] for c in enc.calls] == ["encode_image", "encode_image"] and enc.calls[1][2] == 0.0
    g._prepare_and_encode_inputs([7.0], True)
    assert len(enc.calls) == 3 and list(g.negative_prompt) == ["[NULL_IMAGE]"]      # the negative branch is cached
    enc.calls.clear()
    out = g._prepare_and_encode_inputs(["a cat ", 3.0, " on a mat", 4.0], True)
    assert enc.calls[0] == ("generate_image", ["a cat [<IMG_PLH>] on a mat[<IMG_PLH>]"], (2, 3, 4, 4))
    assert enc.calls[1] == ("generate_image", [""], None)
    assert float(out[0, 0, 0]) == 2.0 and float(out[1, 0, 0]) == -2.0 and set(g.negative_prompt) == {"[NULL_IMAGE]", ""}
    enc.calls.clear()
    out = g._prepare_and_encode_inputs(["only text"], False)
    assert out.shape[0] == 1 and enc.calls == [("generate_image", ["only text"], None)]


def test_chat_forward_batch_builds_one_generate_call():
    """several requests, one EmuModel.generate: texts in request order, pictures concatenated in request order (the order in
    which the <image> slots are filled), one answer per request — each text equal to what `forward` would have sent alone"""
    from PIL import Image
    from emu_b200.emu2.chat import EmuChatGeneration
    fm = _FakeModel()
    fm.generate = lambda **kw: (fm.calls.append(kw), ["answer %d" % i for i in range(len(kw["text"]))])[1]
    fm.engine = type("E", (), {"cfg": type("C", (), {"llm_max_batch": 20})()})()
    pipe = EmuChatGeneration(fm)
    a, b = Image.new("RGB", (30, 20), (255, 0, 0)), Image.new("RGB", (20, 30), (0, 0, 255))
    reqs = [[a, "describe"], ["no picture here"], [["hi", b], ["hello"], ["and?"]]]
    out = pipe.forward_batch(reqs, num_beams=3, max_new_tokens=7)
    assert out == ["answer 0", "answer 1", "answer 2"]
    kw = fm.calls[-1]
    assert kw["num_beams"] == 3 and kw["max_new_tokens"] == 7 and kw["length_penalty"] == -1
    assert kw["image"].shape == (2, 3, 448, 448) and kw["video"] is None
    singles = []
    for r in reqs:
        pipe.forward(r)
        singles.append(fm.calls[-1])
    assert kw["text"] == [s["text"][0] for s in singles]
    assert torch.equal(kw["image"], torch.cat([s["image"] for s in singles if s["image"] is not None]))
    assert pipe.max_requests_per_batch(5) == 4 and pipe.max_requests_per_batch(1) == 20 and pipe.max_requests_per_batch(32) == 1


def test_visual_generation_forward_batch_layout():
    """n requests through one denoise loop: prompt rows [cond_1..cond_n; uncond_1..uncond_n] (the layout emu_denoise_step
    takes), batch_size n, one output per request; without CFG only the cond rows"""
    import numpy as np
    g = _bare_visual_generation()
    seen = {}

    def denoise(prompt_embeds, batch_size, *a, **k):
        seen["embeds"], seen["n"] = prompt_embeds.float(), batch_size
        return torch.zeros(batch_size, 4, 2, 2)
    g.denoise = denoise
    g.decode_latents_uint8 = lambda lat: np.stack([np.full((4, 4, 3), 10 * i, dtype=np.uint8) for i in range(lat.shape[0])])
    g.safety_checker, g._warned_unfiltered = None, True
    outs = g.forward_batch([["a cat"], [5.0], ["a dog ", 2.0]], guidance_scale=3.0)
    assert seen["n"] == 3 and seen["embeds"].shape[0] == 6
    assert seen["embeds"][:, 0, 0].tolist() == [2.0, 1.0, 2.0, -2.0, -1.0, -2.0]   # generation / autoencoding / generation
    assert [o.image.getpixel((0, 0))[0] for o in outs] == [0, 10, 20] and all(o.nsfw_content_detected is None for o in outs)
    g.forward_batch([["a cat"], ["a dog"]], guidance_scale=1.0)
    assert seen["n"] == 2 and seen["embeds"][:, 0, 0].tolist() == [2.0, 2.0]


def test_builtin_diffusion_config_is_the_published_one(tmp_path):
    """`EmuVisualGeneration.from_pretrained(<weights file>)` reads its configuration from the package in the reference
    (Emu2/emu/diffusion.py:254,272); here the published values are built in — same engine configuration either way, and a
    directory overrides them part by part"""
    import ctypes
    import bench
    from emu_b200.emu2 import conf
    from emu_b200.emu2.diffusion import unet_config_from_json, vae_config_from_json

    def raw(struct):
        return ctypes.string_at(ctypes.addressof(struct), ctypes.sizeof(struct))
    unet, vae, sched = conf.load_diffusion_config(None)
    assert unet == conf.EMU2_GEN_UNET and vae == conf.EMU2_GEN_VAE and sched == conf.EMU2_GEN_SCHEDULER
    assert bench.emu2_unet_json() == conf.EMU2_GEN_UNET
    r_unet, r_vae, r_sched = conf.load_diffusion_config(REF_DIFFUSION_CONFIG)
    for mine, ref in ((unet, r_unet), (vae, r_vae), (sched, r_sched)):
        assert all(ref[k] == v for k, v in mine.items())
    assert raw(unet_config_from_json(unet)) == raw(unet_config_from_json(r_unet))
    assert raw(vae_config_from_json(vae)) == raw(vae_config_from_json(r_vae))
    (tmp_path / "scheduler").mkdir()
    json.dump(dict(conf.EMU2_GEN_SCHEDULER, steps_offset=0), open(tmp_path / "scheduler" / "scheduler_config.json", "w"))
    u2, v2, s2 = conf.load_diffusion_config(str(tmp_path))
    assert s2["steps_offset"] == 0 and u2 == conf.EMU2_GEN_UNET and v2 == conf.EMU2_GEN_VAE
