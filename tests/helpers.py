"""Shared test helpers: deterministic reference-format state dicts, tiny configs, a stub tokenizer."""
import hashlib
import math

import torch

TINY_VISION = dict(image_size=56, patch_size=14, width=128, layers=2, head_width=32, mlp_ratio=4.0, n_query=4, v_query=4)
TINY_LLAMA = dict(hidden_size=256, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512,
                  rms_norm_eps=1e-6, max_position_embeddings=512, vocab_size=32000, rope_theta=10000.0)
VOCAB = 32272  # 32000 + [PAD] + 271 Emu2 special tokens (Emu2/emu/lm.py:63)


def _t(gen, shape, std):
    return torch.randn(shape, generator=gen) * std


def make_emu2_state_dict(vision=TINY_VISION, llama=TINY_LLAMA, vocab=VOCAB, seed=0, dtype=torch.float32):
    """Random weights under the reference's key names (SURVEY.md §8b weight contract). Needs no reference code."""
    g = torch.Generator().manual_seed(seed)
    W, L = vision["width"], vision["layers"]
    P = vision["patch_size"]
    G = vision["image_size"] // P
    mlp = int(W * vision["mlp_ratio"])
    sd = {}
    sd["visual.cls_token"] = _t(g, (1, 1, W), 0.05)
    sd["visual.pos_embed"] = _t(g, (1, G * G + 1, W), 0.05)
    sd["visual.patch_embed.proj.weight"] = _t(g, (W, 3, P, P), 0.03)
    sd["visual.patch_embed.proj.bias"] = _t(g, (W,), 0.05)
    for l in range(L):
        p = f"visual.blocks.{l}."
        for n in ("norm1", "norm2"):
            sd[p + n + ".weight"] = 1 + _t(g, (W,), 0.1)
            sd[p + n + ".bias"] = _t(g, (W,), 0.05)
        sd[p + "attn.q_bias"] = _t(g, (W,), 0.05)
        sd[p + "attn.v_bias"] = _t(g, (W,), 0.05)
        sd[p + "attn.qkv.weight"] = _t(g, (3 * W, W), 1 / math.sqrt(W))
        sd[p + "attn.proj.weight"] = _t(g, (W, W), 1 / math.sqrt(W))
        sd[p + "attn.proj.bias"] = _t(g, (W,), 0.05)
        sd[p + "mlp.fc1.weight"] = _t(g, (mlp, W), 1 / math.sqrt(W))
        sd[p + "mlp.fc1.bias"] = _t(g, (mlp,), 0.05)
        sd[p + "mlp.fc2.weight"] = _t(g, (W, mlp), 1 / math.sqrt(mlp))
        sd[p + "mlp.fc2.bias"] = _t(g, (W,), 0.05)
    H, F, NL = llama["hidden_size"], llama["intermediate_size"], llama["num_hidden_layers"]
    sd["decoder.lm.model.embed_tokens.weight"] = _t(g, (vocab, H), 1.0)
    for l in range(NL):
        p = f"decoder.lm.model.layers.{l}."
        for n in ("q_proj", "k_proj", "v_proj", "o_proj"):
            sd[p + f"self_attn.{n}.weight"] = _t(g, (H, H), 1 / math.sqrt(H))
        sd[p + "mlp.gate_proj.weight"] = _t(g, (F, H), 1 / math.sqrt(H))
        sd[p + "mlp.up_proj.weight"] = _t(g, (F, H), 1 / math.sqrt(H))
        sd[p + "mlp.down_proj.weight"] = _t(g, (H, F), 1 / math.sqrt(F))
        sd[p + "input_layernorm.weight"] = 1 + _t(g, (H,), 0.1)
        sd[p + "post_attention_layernorm.weight"] = 1 + _t(g, (H,), 0.1)
    sd["decoder.lm.model.norm.weight"] = 1 + _t(g, (H,), 0.1)
    sd["decoder.lm.lm_head.weight"] = _t(g, (vocab, H), 1 / math.sqrt(H))
    sd["project_up.weight"] = _t(g, (H, W), 1 / math.sqrt(W))
    sd["project_down.weight"] = _t(g, (W, H), 1 / math.sqrt(H))
    return {k: v.to(dtype) for k, v in sd.items()}


PARITY_RATIO = 1.5   # engine error vs the fp32 reference, in units of what bf16 storage costs the reference itself
PARITY_FLOOR = 2e-3   # half a bf16 ulp of the largest element: below this the two rounding-noise samples are not comparable


def bf16_state_dict(sd):
    return {k: v.to(torch.bfloat16) for k, v in sd.items()}


def assert_bf16_parity(name, out, ref32, ref16, ratio=PARITY_RATIO, floor=PARITY_FLOOR):
    """The parity bound used by every model-level GPU test (VERDICT r01 item 1b): the engine keeps activations in bf16 exactly
    where the reference's own bf16 run rounds, so its distance from the fp32 reference must not exceed `ratio` x the distance
    of the CPU oracle run in the same dtype policy (ref16) — no hard-coded budget.  Returns (engine error, bf16-oracle error)."""
    from oracle import emu_oracle as O
    e_eng, e_bf = O.rel_err(out, ref32), O.rel_err(ref16, ref32)
    print("\n[parity] %-34s engine-vs-fp32 %.3e | bf16-oracle-vs-fp32 %.3e | ratio %.2f" % (name, e_eng, e_bf, e_eng / max(e_bf, 1e-12)))
    assert e_eng <= max(ratio * e_bf, floor), (name, e_eng, e_bf)
    return e_eng, e_bf


def tensor_digest(t, n_sample=512):
    """Stand-in for a tensor too large to store as a golden fixture: shape, dtype, the SHA-256 of its bytes and a seeded
    sample of its values (the sample makes a mismatch readable; the hash keeps the comparison bit-exact)."""
    t = t.detach().contiguous().cpu()
    flat = t.reshape(-1)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:n_sample].clone()
    return {"shape": tuple(t.shape), "dtype": str(t.dtype), "sha256": hashlib.sha256(t.numpy().tobytes()).hexdigest(),
            "idx": idx, "sample": flat[idx].clone()}


def assert_equal_digest(t, d):
    """`t` is bitwise equal to the tensor `d` = tensor_digest(...) was made from."""
    t = t.detach().contiguous().cpu()
    assert tuple(t.shape) == d["shape"] and str(t.dtype) == d["dtype"], (tuple(t.shape), t.dtype, d["shape"], d["dtype"])
    s = t.reshape(-1)[d["idx"]]
    assert torch.equal(s, d["sample"]), "max |diff| on the sampled values: %g" % (s - d["sample"]).abs().max()
    assert hashlib.sha256(t.numpy().tobytes()).hexdigest() == d["sha256"]


def chat_prompt_cases():
    """Inputs of the chat prompt-assembly comparison (tests/test_host_cpu.py, tests/golden/gen_golden_reference_checks.py):
    plain messages for _prepare_inputs and (conversation, is_grounding) pairs for _prepare_chat_inputs."""
    from PIL import Image
    from emu_b200.emu2.constants import DEFAULT_VIDEO_TOKEN, FAKE_VIDEO_END_TOKEN
    imgs = [Image.new("RGB", (64 + 10 * i, 48 + 7 * i), (10 * i, 200 - 20 * i, 30 + i)) for i in range(4)]
    plain = [
        [imgs[0], "describe"],
        ["before", imgs[1], "between", imgs[2], "after"],
        ["watch:", DEFAULT_VIDEO_TOKEN, imgs[0], imgs[1], FAKE_VIDEO_END_TOKEN, "what happens?", imgs[3]],
        ["text only"],
    ]
    chats = [
        ([[imgs[0], "what is this?"], ["a cat"], ["and this?", imgs[1]]], True),
        ([["hello"]], False),
        ([[imgs[2], imgs[3], "compare"], ["they differ"], ["how?"]], False),
    ]
    return plain, chats


class StubTokenizer:
    """Just enough of the HF tokenizer surface for EmuModel when texts are pre-tokenised (GPU box has no
    tokenizer.model: the reference's file is not redistributed; golden fixtures carry the real ids)."""
    pad_token_id, bos_token_id, eos_token_id = 32000, 1, 2
    padding_side = truncation_side = "left"
    _special = {"[IMG]": 32001, "[/IMG]": 32002, "<image>": 32003, "[gIMG]": 32004}

    def __len__(self):
        return VOCAB

    def convert_tokens_to_ids(self, toks):
        return [self._special[t] for t in toks]

    def batch_decode(self, ids, skip_special_tokens=True):
        return [" ".join(str(int(i)) for i in row if not (skip_special_tokens and int(i) in (0, 1, 2, 32000))) for row in ids]


# ---- Emu1 fixtures (shared by tests/test_emu1_vae_gpu.py and tests/golden/gen_golden_emu1.py) ----
EMU1_VIS = dict(image_size=56, patch_size=14, width=128, layers=2, head_width=32, mlp_ratio=4.0)  # head_dim 32
EMU1_VIS88 = dict(image_size=56, patch_size=14, width=176, layers=2, head_width=88, mlp_ratio=4.0)  # head_dim 88 like EVA-g
EMU1_LLAMA = dict(hidden_size=256, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512, rms_norm_eps=1e-6,
                  max_position_embeddings=256, vocab_size=32000, rope_theta=10000.0)


def emu1_t5_cfg():
    from oracle import t5_oracle as T
    return dict(T.T5_BASE, layers=2, d_model=128, heads=2, d_ff=256)


def emu1_state_dict(vis, seed=0):
    from oracle import diffusion_oracle as D
    from oracle import t5_oracle as T
    sd = make_emu2_state_dict(vision=dict(vis, n_query=4, v_query=4), llama=EMU1_LLAMA, vocab=32004, seed=seed)
    sd.pop("project_up.weight"), sd.pop("project_down.weight")
    g = torch.Generator().manual_seed(seed + 100)
    W = vis["width"]
    sd["ln_visual.weight"] = 1 + 0.1 * torch.randn(W, generator=g)
    sd["ln_visual.bias"] = 0.05 * torch.randn(W, generator=g)
    sd["decoder.lm.stu_regress_head.weight"] = torch.randn(256, 256, generator=g) / 16
    cf = D.random_state_dict(T.param_shapes(emu1_t5_cfg(), W, 256, n_causal=8), seed=seed + 7)
    for k in cf:  # T5 attention is unscaled: the Mesh-TF init keeps q small so that the softmax is not saturated
        if k.endswith("Attention.q.weight"):
            cf[k] = cf[k] * 0.125
    sd.update(cf)
    return sd
