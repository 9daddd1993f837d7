"""CPU: the oracle restatement (oracle/emu_oracle.py) against the golden outputs of the UNMODIFIED reference
(tests/golden/emu2_tiny.pt, made by tests/golden/gen_golden.py; tests/golden/reference_checks.pt, made by
tests/golden/gen_golden_reference_checks.py)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import TINY_LLAMA, make_emu2_state_dict
from oracle import emu_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "emu2_tiny.pt")
L, NH = TINY_LLAMA["num_hidden_layers"], TINY_LLAMA["num_attention_heads"]


@pytest.fixture(scope="module")
def gold():
    return torch.load(GOLD)


@pytest.fixture(scope="module")
def sd():
    return make_emu2_state_dict()


def test_vit_and_encode_image(gold, sd):
    f = O.vit_forward_features(sd, gold["image"], patch=14, num_heads=4, layers=2)
    assert O.rel_err(f, gold["vit_tokens"]) < 1e-5
    e = O.encode_image(sd, gold["image"], patch=14, num_heads=4, layers=2, n_query=4)
    assert O.rel_err(e, gold["encode_image"]) < 1e-5


def _prompt_embeds(gold, sd):
    e = O.encode_image(sd, gold["image"], patch=14, num_heads=4, layers=2, n_query=4)
    pie = F.linear(e.view(-1, e.shape[-1]), sd["project_up.weight"])
    return O.splice_embeds(sd, gold["gen_input_ids"], pie, 32003)


def test_prefill_logits(gold, sd):
    emb = _prompt_embeds(gold, sd)
    mask = gold["gen_attention_mask"]
    h = O.llama_forward(sd, emb, mask, layers=L, heads=NH, position_ids=O.hf_position_ids(mask))
    assert O.rel_err(O.lm_logits(sd, h[:, -1]), gold["prefill_logits_last"]) < 1e-4


def test_greedy_tokens(gold, sd):
    toks = O.generate_greedy(sd, _prompt_embeds(gold, sd), gold["gen_attention_mask"], layers=L, heads=NH,
                             max_new_tokens=12, min_len=1)
    assert torch.equal(toks, gold["gen_ids_greedy"])


def test_generate_image_literal_and_cached(gold, sd):
    ids, mask = gold["genimg_input_ids"], gold["genimg_attention_mask"]
    pe = F.embedding(ids, sd["decoder.lm.model.embed_tokens.weight"])
    out = O.generate_image_cached(sd, pe, mask, 4, layers=L, heads=NH)
    assert O.rel_err(out, gold["genimg_text"]) < 1e-4
    # multimodal prompt: prompt-image slots filled with project_up(encode_image)
    ids2, mask2 = gold["genimg_mm_input_ids"], gold["genimg_mm_attention_mask"]
    e = O.encode_image(sd, gold["image"][:1], patch=14, num_heads=4, layers=2, n_query=4)
    pe2 = O.splice_embeds(sd, ids2, F.linear(e.view(-1, e.shape[-1]), sd["project_up.weight"]), 32003)
    out2 = O.generate_image_cached(sd, pe2, mask2, 4, layers=L, heads=NH)
    assert O.rel_err(out2, gold["genimg_mm"]) < 1e-4


@pytest.fixture(scope="module")
def ref_checks():
    return torch.load(os.path.join(os.path.dirname(GOLD), "reference_checks.pt"))


def test_oracle_vs_live_reference(sd, ref_checks):
    """encode_image and the literal generate_image against the outputs of the UNMODIFIED reference EmuModel on the same
    weights, fed the ids its own tokenizer produced (tests/golden/gen_golden_reference_checks.py)"""
    ref = ref_checks["emu2_tiny"]
    img = torch.randn(1, 3, 56, 56, generator=torch.Generator().manual_seed(5))
    assert O.rel_err(O.encode_image(sd, img, patch=14, num_heads=4, layers=2, n_query=4), ref["encode_image"]) < 1e-5
    lit = O.generate_image_regress(sd, lambda k: ref["generate_image_ids"][k], 4, layers=L, heads=NH, image_token_id=32003,
                                   boi_token_id=32001)
    assert O.rel_err(lit, ref["generate_image"]) < 1e-5


@pytest.mark.parametrize("H,W,S", [(37, 53, 16), (500, 333, 448), (448, 448, 448), (1024, 768, 448), (100, 100, 224),
                                   (31, 97, 224), (224, 1000, 448)])
def test_preprocess_oracle_vs_torchvision(H, W, S):
    """oracle/preprocess_oracle.py must be BIT-EXACT with the reference's own transform (Emu2/emu/chat.py:35-39:
    torchvision Resize(BICUBIC) on a PIL image -> ToTensor -> Normalize), up- and down-scaling, ragged sizes."""
    tv = pytest.importorskip("torchvision.transforms")
    from PIL import Image
    from oracle import preprocess_oracle as P
    mean, std = (0.48145466, 0.4578275, 0.40821073), (0.26862954, 0.26130258, 0.27577711)
    rng = np.random.default_rng(H * 1000 + W)
    img = (rng.random((H, W, 3)) * 255).astype(np.uint8)
    pil = Image.fromarray(img)
    assert np.array_equal(np.asarray(pil.resize((S, S), Image.BICUBIC)), P.resize_bicubic_u8(img, S, S))
    t = tv.Compose([tv.Resize((S, S), interpolation=tv.InterpolationMode.BICUBIC), tv.ToTensor(),
                    tv.Normalize(mean=mean, std=std)])
    assert np.array_equal(t(pil).numpy(), P.image_transform(img, S, mean, std))


def _cformer_state_dict(g):
    """the seeded Causal-Former weights a golden file was made with"""
    from oracle import diffusion_oracle as D, t5_oracle as T
    sd = D.random_state_dict(T.param_shapes(g["cfg"], g["enc_w"], g["out_dim"], n_causal=g["n_causal"]), seed=g["seed"])
    for k in sd:
        if k.endswith("Attention.q.weight"):
            sd[k] = sd[k] * 0.125
    return sd


def _cformer_golden():
    g = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "emu1_cformer_tiny.pt"))
    return g, _cformer_state_dict(g)


def test_t5_oracle_vs_reference_golden():
    """oracle/t5_oracle.py (Causal-Former restatement) reproduces the outputs the UNMODIFIED reference module produced
    (tests/golden/gen_golden_cformer.py) bit for bit, fp32 and bf16."""
    from oracle import t5_oracle as T
    g, sd = _cformer_golden()
    out = T.causal_former(sd, g["img_embeds"], g["cfg"])
    assert torch.equal(out, g["out_fp32"])
    sd16 = {k: v.to(torch.bfloat16) for k, v in sd.items()}
    out16 = T.causal_former(sd16, g["img_embeds"].to(torch.bfloat16), g["cfg"]).float()
    assert torch.equal(out16, g["out_bf16"])


def test_t5_oracle_vs_live_reference_t5_base(ref_checks):
    """Same, at the real t5-base dimensions (12 layers, d_model 768, 32 causal queries over 257 EVA-CLIP tokens of width
    1408): the outputs the reference module produced on seeded weights (tests/golden/gen_golden_reference_checks.py) —
    bit-exact, fp32 and bf16."""
    from oracle import t5_oracle as T
    g = ref_checks["t5_base"]
    assert g["cfg"] == T.T5_BASE
    sd = _cformer_state_dict(g)
    x = torch.randn(*g["img_embeds_shape"], generator=torch.Generator().manual_seed(g["seed"] + 1))
    threads = torch.get_num_threads()
    torch.set_num_threads(1)   # at these widths the CPU GEMMs split their sums by thread count: one thread, as the golden run
    try:
        for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
            sdt = {k: v.to(dt) for k, v in sd.items()}
            assert torch.equal(T.causal_former(sdt, x.to(dt)), g["out_" + name]), name
    finally:
        torch.set_num_threads(threads)


def test_emu1_oracle_vs_reference_golden():
    """Emu1 image path of the oracle (pre-norm EVA ViT -> ln_visual -> Causal-Former) == outputs of the UNMODIFIED
    reference modules (tests/golden/gen_golden_emu1.py), bit for bit, head widths 32 and 88."""
    from helpers import EMU1_VIS, EMU1_VIS88, emu1_state_dict, emu1_t5_cfg
    from oracle import t5_oracle as T
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "emu1_tiny.pt"))
    for vis in (EMU1_VIS, EMU1_VIS88):
        g = gold["w%d" % vis["width"]]
        sd = emu1_state_dict(vis)
        feats = O.vit_forward_features(sd, g["image"], patch=14, num_heads=vis["width"] // vis["head_width"], layers=2,
                                       postnorm=False)
        feats = F.layer_norm(feats, (vis["width"],), sd["ln_visual.weight"], sd["ln_visual.bias"], 1e-6)
        assert torch.equal(feats, g["ln_visual_features"])
        assert torch.equal(T.causal_former(sd, feats, emu1_t5_cfg()), g["cformer_out"])


def test_emu1_vit_oracle_vs_live_reference(ref_checks):
    """the pre-norm EVA ViT at head width 88 == forward_features of the reference's EVAVisionTransformer on the same seeded
    weights (tests/golden/gen_golden_reference_checks.py), bit for bit"""
    from helpers import EMU1_VIS88, emu1_state_dict
    sd = emu1_state_dict(EMU1_VIS88)
    img = torch.randn(2, 3, 56, 56, generator=torch.Generator().manual_seed(9))
    assert torch.equal(ref_checks["emu1_vit88"]["forward_features"],
                       O.vit_forward_features(sd, img, patch=14, num_heads=2, layers=2, postnorm=False))


def _emu1_generate_image_oracle(sd, ids, image, vis):
    """Emu1/models/modeling_emu.py:187-249 restated with the oracle pieces (cache-less literal loop: every iteration
    re-runs the decoder over the grown sequence and appends stu_regress_head(h_last))."""
    from helpers import emu1_t5_cfg
    from oracle import t5_oracle as T
    emb = F.embedding(ids, sd["decoder.lm.model.embed_tokens.weight"])
    if image is not None:
        feats = O.vit_forward_features(sd, image, patch=14, num_heads=vis["width"] // vis["head_width"], layers=2, postnorm=False)
        feats = F.layer_norm(feats, (vis["width"],), sd["ln_visual.weight"], sd["ln_visual.bias"], 1e-6)
        cf = T.causal_former(sd, feats, emu1_t5_cfg())
        emb[ids == 32003] = cf.reshape(-1, cf.shape[-1])
    outs = []
    for _ in range(8):
        h = O.llama_forward(sd, emb, torch.ones(1, emb.shape[1], dtype=torch.long), layers=2, heads=2)
        reg = F.linear(h[:, -1], sd["decoder.lm.stu_regress_head.weight"])
        outs.append(reg)
        emb = torch.cat((emb, reg[:, None]), dim=1)
    return torch.stack(outs, dim=1)


def test_emu1_generate_image_oracle_vs_reference_golden():
    """The oracle's Emu1 generate_image == the UNMODIFIED reference `Emu.generate_image` (tests/golden/
    gen_golden_emu1_genimg.py; its own tokenizer, 8 full re-forwards), text-only and with a prompt image."""
    from helpers import EMU1_VIS, emu1_state_dict
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "emu1_genimg_tiny.pt"))
    sd = emu1_state_dict(EMU1_VIS)
    for key in ("text_only", "with_image"):
        g = gold[key]
        out = _emu1_generate_image_oracle(sd, g["input_ids"], g.get("image"), EMU1_VIS)
        assert out.shape == g["embeds"].shape
        assert O.rel_err(out, g["embeds"]) < 1e-5, (key, O.rel_err(out, g["embeds"]))
