"""GPU: checkpoint ingestion END TO END (SURVEY.md §8f-3) — a model file in each reference format, streamed tensor by tensor into
the engine by emu_b200/checkpoint.py, must give the engine the same weights as handing it the state dict directly: the
image tokens and the first-step logits are compared BITWISE.  Formats: a single safetensors file, a torch .bin, an HF sharded
index (Emu2/emu/conf/llama_config/pytorch_model.bin.index.json style), the Emu1 `{"module": ...}` wrapper, and LoRA adapters in
the peft key layout merged while streaming (Emu1/inference.py:40-57)."""
import json
import os

import pytest
import torch

from helpers import TINY_LLAMA, TINY_VISION, StubTokenizer, make_emu2_state_dict

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "emu2_tiny.pt")


def _model():
    from emu_b200.emu2.conf import CLIPVisionCfg, TextDecoderCfg
    from emu_b200.emu2.emu import EmuModel
    return EmuModel(CLIPVisionCfg(**TINY_VISION), TextDecoderCfg(), tokenizer=StubTokenizer(), llama_config=TINY_LLAMA,
                    max_batch=2, max_seq=64)


def _outputs(m, gold):
    ids, mask = gold["gen_input_ids"].cuda(), gold["gen_attention_mask"].cuda()
    e = m.encode_image(gold["image"].cuda())
    emb = m.engine.llm_embed(ids)
    emb[ids == 32003] = m._project_up(e.reshape(-1, e.shape[-1]))
    m.engine.llm_reset()
    _, logits = m.engine.llm_prefill(emb, mask, hf_positions=True, want_logits=True)
    return e.float().cpu(), logits.cpu()


@pytest.fixture(scope="module")
def want(cuda):
    gold = torch.load(GOLD)
    sd = {k: v.to(torch.bfloat16) for k, v in make_emu2_state_dict().items()}
    m = _model()
    m.load_state_dict(sd)
    return gold, sd, _outputs(m, gold)


def _write(fmt, sd, d):
    from safetensors.torch import save_file
    if fmt == "safetensors":
        p = os.path.join(d, "model.safetensors")
        save_file({k: v.contiguous() for k, v in sd.items()}, p)
        return p
    if fmt == "bin":
        p = os.path.join(d, "pytorch_model.bin")
        torch.save(sd, p)
        return p
    if fmt == "module":
        p = os.path.join(d, "emu1_style.pt")
        torch.save({"module": sd}, p)
        return p
    assert fmt == "sharded"
    keys = sorted(sd)
    cut = [keys[i::3] for i in range(3)]
    wm = {}
    for i, ks in enumerate(cut):
        name = "pytorch_model-%05d-of-00003.bin" % (i + 1)
        torch.save({k: sd[k] for k in ks}, os.path.join(d, name))
        wm.update({k: name for k in ks})
    json.dump({"metadata": {}, "weight_map": wm}, open(os.path.join(d, "pytorch_model.bin.index.json"), "w"))
    return d


@pytest.mark.parametrize("fmt", ["safetensors", "bin", "module", "sharded"])
def test_checkpoint_file_equals_state_dict(want, tmp_path, fmt):
    from emu_b200 import checkpoint
    gold, sd, (e0, l0) = want
    m = _model()
    n = checkpoint.load_into(m.engine, _write(fmt, sd, str(tmp_path)))
    assert n == len(sd)
    e1, l1 = _outputs(m, gold)
    assert torch.equal(e0, e1) and torch.equal(l0, l1)


def test_lora_adapters_are_merged_while_streaming(want, tmp_path):
    """q_proj of layer 0 saved as base + (B @ A) * alpha / r in the peft layout == the merged weight saved plainly"""
    from emu_b200 import checkpoint
    gold, sd, _ = want
    key = "decoder.lm.model.layers.0.self_attn.q_proj"
    g = torch.Generator().manual_seed(5)
    r = 4
    A = (torch.randn(r, sd[key + ".weight"].shape[1], generator=g) * 0.05).to(torch.bfloat16)
    B = (torch.randn(sd[key + ".weight"].shape[0], r, generator=g) * 0.05).to(torch.bfloat16)
    lora_sd = {k: v for k, v in sd.items() if k != key + ".weight"}
    lora_sd[key + ".base_layer.weight"] = sd[key + ".weight"]
    lora_sd[key + ".lora_A.default.weight"], lora_sd[key + ".lora_B.default.weight"] = A, B
    torch.save(lora_sd, str(tmp_path / "lora.bin"))
    seen = {}

    class Tap:                                    # what the loader hands the engine for that key
        def load_tensor(self, k, t):
            seen[k] = t.clone()
    checkpoint.load_into(Tap(), str(tmp_path / "lora.bin"), lora=True)
    merged = dict(sd)
    merged[key + ".weight"] = seen[key + ".weight"]
    assert not torch.equal(merged[key + ".weight"], sd[key + ".weight"])
    ma, mb = _model(), _model()
    checkpoint.load_into(ma.engine, str(tmp_path / "lora.bin"), lora=True)
    mb.load_state_dict(merged)
    (ea, la), (eb, lb) = _outputs(ma, gold), _outputs(mb, gold)
    assert torch.equal(ea, eb) and torch.equal(la, lb)
