"""Generate tests/golden/emu2_tiny.pt by running the UNMODIFIED reference (/root/reference/Emu2/emu) on CPU.

Run in the authoring container only:  python tests/golden/gen_golden.py
The fixture carries the reference's own outputs (fp32) for a tiny configuration plus the real tokenizer's ids, so
the GPU box — which has neither /root/reference nor tokenizer.model — can check the CUDA path against the reference.
Weights are regenerated on the box from tests/helpers.make_emu2_state_dict(seed=0).
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import TINY_LLAMA, TINY_VISION, make_emu2_state_dict  # noqa: E402
from oracle import ref_shim  # noqa: E402


def main():
    torch.manual_seed(0)
    d = ref_shim.make_llama_config_dir(TINY_LLAMA["hidden_size"], TINY_LLAMA["num_hidden_layers"],
                                       TINY_LLAMA["num_attention_heads"], TINY_LLAMA["intermediate_size"],
                                       max_pos=TINY_LLAMA["max_position_embeddings"])
    vk = dict(TINY_VISION)
    vk.pop("patch_size")
    model = ref_shim.build_emu2_model(dict(vk, patch_size=14), d)
    sd = make_emu2_state_dict()
    model.load_state_dict(sd, strict=True)  # the reference's own strict load (Emu2/emu/chat.py:212)
    tok = model.decoder.tokenizer
    g = torch.Generator().manual_seed(1234)
    image = torch.randn(2, 3, 56, 56, generator=g)
    out = {"image": image}
    with torch.no_grad():
        out["vit_tokens"] = model.visual(image)
        out["encode_image"] = model.encode_image(image)
        texts = ["[<IMG_PLH>]Describe the image in details:", "[<IMG_PLH>]What is shown? Please answer:"]
        t2 = [t.replace("[<IMG_PLH>]", model.image_placeholder) for t in texts]
        inp = tok(t2, padding="longest", return_tensors="pt")
        out["gen_input_ids"], out["gen_attention_mask"] = inp.input_ids, inp.attention_mask
        # first-step logits of the reference's own LlamaForCausalLM on the spliced embeddings
        emb = model.decoder.lm.model.embed_tokens(inp.input_ids)
        pe = model.project_up(out["encode_image"].view(-1, TINY_VISION["width"]))
        emb[inp.input_ids == 32003] = pe
        pos = (inp.attention_mask.cumsum(-1) - 1).masked_fill(inp.attention_mask == 0, 1)
        lo = model.decoder.lm(inputs_embeds=emb, attention_mask=inp.attention_mask, position_ids=pos)
        out["prefill_logits_last"] = lo.logits[:, -1, :].float().clone()   # own storage: a view saves all [B, T, vocab] logits
        # generate: new-token ids straight from lm.generate (what EmuModel.generate decodes, emu.py:213-233)
        from emu.emu import GENERATION_CONFIG
        for name, kw in (("greedy", dict(num_beams=1)), ("beam5", dict(num_beams=5, length_penalty=-1)),
                         ("beam3_lp1", dict(num_beams=3, length_penalty=1.0))):
            B = 1 if kw["num_beams"] == 5 else 2
            ids = model.decoder.lm.generate(generation_config=GENERATION_CONFIG, inputs_embeds=emb[:B],
                                            attention_mask=inp.attention_mask[:B], do_sample=False,
                                            max_new_tokens=12, min_length=1, repetition_penalty=1.0, **kw)
            out["gen_ids_" + name] = ids
            out["gen_text_" + name] = tok.batch_decode(ids, skip_special_tokens=True)
        # end-to-end through the reference API as a cross-check of the splice logic
        out["gen_text_api_greedy"] = model.generate(text=texts, image=image, num_beams=1, max_new_tokens=12)
        # generate_image (text only and text + image prompt)
        gtexts = ["a photo of a cat", "an astronaut riding a horse on mars"]
        out["genimg_text"] = model.generate_image(text=gtexts)
        gi = tok([t + "[IMG]" for t in gtexts], padding="longest", return_tensors="pt")
        out["genimg_input_ids"], out["genimg_attention_mask"] = gi.input_ids, gi.attention_mask
        g2 = ["[<IMG_PLH>]make it blue"]
        out["genimg_mm"] = model.generate_image(text=g2, image=image[:1])
        gi2 = tok([t.replace("[<IMG_PLH>]", model.image_placeholder) + "[IMG]" for t in g2], padding="longest",
                  return_tensors="pt")
        out["genimg_mm_input_ids"], out["genimg_mm_attention_mask"] = gi2.input_ids, gi2.attention_mask
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu2_tiny.pt")
    torch.save(out, path)
    print("wrote", path, {k: (tuple(v.shape) if hasattr(v, "shape") else v) for k, v in out.items()})


if __name__ == "__main__":
    main()
