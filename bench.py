#!/usr/bin/env python
"""bench.py — headline benchmark of the Emu2 image->text generate path on B200 (BASELINE.json configs[1]).

One "step" = one full pass of the hot path over one synthetic request: 1x448x448 image -> EVA-CLIP-4B ViT ->
project_up -> splice into the ~75-token prompt -> LLaMA-33B prefill -> 128 greedily decoded tokens (EOS suppressed so
exactly 128 steps run).  bf16 weights/activations, random-init weights of the real architecture, synthetic image/ids.

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA engine (tensor parallel for N > 1)
  python bench.py --impl reference ...                   # the reference's CPU path, bounded sample (rank 0 only)
  python bench.py ... --dump-outputs DIR                 # also write the last timed step's outputs as DIR/<name>.npy

Prints ONE JSON line (see the task contract): value = device-resident tok/s, e2e = through the public API with host
buffers, roofline = achieved HBM GB/s of the decode step's weight-streaming kernels vs MEASURED_PEAKS.json,
cpu_baseline = the oracle port timed on this box's host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "emu2_img2text_decode_tok_per_s"
NEW_TOKENS = 128
N_TEXT = 8


def emu2_cfgs(small=False):
    from emu_b200.emu2.conf import CLIPVisionCfg, EMU2_LLAMA_33B
    if small:  # plumbing-only configuration for CPU-side dry runs of this script's logic (never reported)
        return CLIPVisionCfg(image_size=56, width=128, layers=2, head_width=32, mlp_ratio=4.0, n_query=4), dict(
            hidden_size=256, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512, rms_norm_eps=1e-6,
            max_position_embeddings=512, vocab_size=32000, rope_theta=10000.0)
    return CLIPVisionCfg(), dict(EMU2_LLAMA_33B)


def llm_bytes_per_token(lc, vocab):
    """Algorithmic HBM bytes one decoded token must read at batch 1 (SURVEY.md §8d): all decoder weights + lm_head."""
    H, F, L = lc["hidden_size"], lc["intermediate_size"], lc["num_hidden_layers"]
    per_layer = 4 * H * H + 3 * H * F + 2 * H
    return 2 * (L * per_layer + H + vocab * H)


def kv_bytes_per_ctx_token(lc):
    return 2 * lc["num_hidden_layers"] * lc["hidden_size"] * 2


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx.append(float(p[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write what the timed path returned in its last step as <out_dir>/<name>.npy — floating-point results as float32,
    token ids as float64 (exact) — so that two builds can be compared output for output on the same seeded inputs."""
    import numpy as np
    host = {name: (t.float() if t.is_floating_point() else t.double()).cpu().numpy() for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# reference / cpu_baseline arm: the oracle port of the reference's CPU path on a bounded sample
# ------------------------------------------------------------------------------------------------
_CPU_SD_CACHE = {}


_CPU_BEST_THREADS = None
_CPU_KIND = "port"   # "reference" once the LLaMA part of the CPU arm ran through transformers' own LlamaForCausalLM


def ncu_traffic():
    """dram bytes / algorithmic bytes of the dominant kernel, from the ncu --set full capture committed this round
    (profiles/r02_ncu_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep of the gate/up GEMV launch)."""
    for name in ("r02_ncu_traffic.json",):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            try:
                d = json.load(open(p))
                return float(d["dram_bytes_per_launch"]) / float(d["algorithmic_bytes_per_launch"]), "profiles/" + name
            except Exception:
                pass
    return None, None


def _cpu_state(lc, vc, vocab, layers_sampled, g):
    """Random-init real-shape weights of `layers_sampled` LLaMA layers + lm_head and ONE EVA-CLIP block (bf16, host)."""
    H, F = lc["hidden_size"], lc["intermediate_size"]
    key = (H, F, vocab, layers_sampled, vc.width)
    if key in _CPU_SD_CACHE:
        return _CPU_SD_CACHE[key]
    sd = {}
    rn = lambda *sh: (torch.randn(*sh, generator=g) * 0.02).to(torch.bfloat16)
    for l in range(layers_sampled):
        p = f"decoder.lm.model.layers.{l}."
        for n in ("q_proj", "k_proj", "v_proj", "o_proj"):
            sd[p + f"self_attn.{n}.weight"] = rn(H, H)
        sd[p + "mlp.gate_proj.weight"] = rn(F, H)
        sd[p + "mlp.up_proj.weight"] = rn(F, H)
        sd[p + "mlp.down_proj.weight"] = rn(H, F)
        sd[p + "input_layernorm.weight"] = torch.ones(H, dtype=torch.bfloat16)
        sd[p + "post_attention_layernorm.weight"] = torch.ones(H, dtype=torch.bfloat16)
    sd["decoder.lm.model.norm.weight"] = torch.ones(H, dtype=torch.bfloat16)
    sd["decoder.lm.lm_head.weight"] = rn(vocab, H)
    W, M = vc.width, int(vc.width * vc.mlp_ratio)
    v = "visual.blocks.0."
    sd[v + "attn.qkv.weight"] = rn(3 * W, W)
    sd[v + "attn.q_bias"] = rn(W)
    sd[v + "attn.v_bias"] = rn(W)
    sd[v + "attn.proj.weight"] = rn(W, W)
    sd[v + "attn.proj.bias"] = rn(W)
    sd[v + "mlp.fc1.weight"] = rn(M, W)
    sd[v + "mlp.fc1.bias"] = rn(M)
    sd[v + "mlp.fc2.weight"] = rn(W, M)
    sd[v + "mlp.fc2.bias"] = rn(W)
    for n in ("norm1", "norm2"):
        sd[v + n + ".weight"] = torch.ones(W, dtype=torch.bfloat16)
        sd[v + n + ".bias"] = torch.zeros(W, dtype=torch.bfloat16)
    _CPU_SD_CACHE[key] = sd
    return sd


def _llama_cpu_times_port(lc, layers_sampled, sd, ctx, tokens, threads, budget_s, g):
    """-> (prefill seconds for all layers, [(per-layer s, head s)] per timed token, label) via oracle/emu_oracle.py"""
    from oracle import emu_oracle as O
    H, nh = lc["hidden_size"], lc["num_attention_heads"]
    cache = O.KVCache(layers_sampled)
    torch.set_num_threads(os.cpu_count())
    x = (torch.randn(1, ctx, H, generator=g) * 0.02).to(torch.bfloat16)
    mask = torch.ones(1, ctx, dtype=torch.long)
    O.llama_forward(sd, x, mask, layers=layers_sampled, heads=nh, cache=O.KVCache(layers_sampled))
    t0 = time.perf_counter()
    O.llama_forward(sd, x, mask, layers=layers_sampled, heads=nh, cache=cache)
    prefill_s = (time.perf_counter() - t0) * lc["num_hidden_layers"] / layers_sampled
    torch.set_num_threads(threads)
    per_tok = []
    t_start = time.time()
    for i in range(tokens + 1):
        e = (torch.randn(1, 1, H, generator=g) * 0.02).to(torch.bfloat16)
        mask = torch.cat((mask, torch.ones(1, 1, dtype=torch.long)), dim=1)
        t0 = time.perf_counter()
        h = O.llama_forward(sd, e, mask, layers=layers_sampled, heads=nh, cache=cache, final_norm=False)
        t1 = time.perf_counter()
        hn = O.rms_norm(h, sd["decoder.lm.model.norm.weight"], 1e-6)
        O.lm_logits(sd, hn[:, -1]).float().argmax(-1)
        t2 = time.perf_counter()
        if i > 0:  # first step is warm-up
            per_tok.append(((t1 - t0) / layers_sampled, t2 - t1))
        if time.time() - t_start > budget_s and len(per_tok) >= 1:
            break
    return prefill_s, per_tok, "oracle/emu_oracle.py (port of HF LlamaDecoderLayer)"


def _llama_cpu_times_hf(lc, vocab, layers_sampled, sd, ctx, tokens, threads, budget_s, g):
    """Same measurement through transformers' own `LlamaForCausalLM` (eager attention, bf16, KV cache) — the module the reference
    builds in Emu2/emu/lm.py:38 and drives through `lm.generate(inputs_embeds=...)` — with `layers_sampled` layers at the real
    width, sharing the weight tensors of `sd`.  Decoder-layer times come from forward hooks (they do not change the
    computation); what is left of a step (final norm, lm_head, cache / mask plumbing) is the per-token head time."""
    import transformers
    from transformers import LlamaConfig, LlamaForCausalLM
    from transformers.cache_utils import DynamicCache
    from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding
    H, nh = lc["hidden_size"], lc["num_attention_heads"]
    cfg = LlamaConfig(hidden_size=H, intermediate_size=lc["intermediate_size"], num_hidden_layers=layers_sampled,
                      num_attention_heads=nh, num_key_value_heads=nh, vocab_size=vocab, rms_norm_eps=lc["rms_norm_eps"],
                      max_position_embeddings=lc.get("max_position_embeddings", 2048), rope_theta=lc.get("rope_theta", 10000.0),
                      attn_implementation="eager")
    with torch.device("meta"):                     # no second copy of the weights: the parameters ARE the tensors of `sd`
        model = LlamaForCausalLM(cfg).to(torch.bfloat16)
    mapped = {k[len("decoder.lm."):]: v for k, v in sd.items() if k.startswith("decoder.lm.")}
    missing, unexpected = model.load_state_dict(mapped, assign=True, strict=False)
    if unexpected or set(missing) - {"model.embed_tokens.weight"}:     # inputs_embeds drive it: the embedding table is not used
        raise RuntimeError("state dict does not fit LlamaForCausalLM: missing %s unexpected %s" % (missing, unexpected))
    model.model.rotary_emb = LlamaRotaryEmbedding(cfg)                  # its inv_freq buffer was created on the meta device
    model.eval()
    layer_t = []

    def pre(mod, a, k):
        mod._t0 = time.perf_counter()

    def post(mod, a, k, out):
        layer_t.append(time.perf_counter() - mod._t0)
    for layer in model.model.layers:
        layer.register_forward_pre_hook(pre, with_kwargs=True)
        layer.register_forward_hook(post, with_kwargs=True)

    def step(x, mask, cache):
        layer_t.clear()
        t0 = time.perf_counter()
        out = model(inputs_embeds=x, attention_mask=mask, past_key_values=cache, use_cache=True, logits_to_keep=1)
        out.logits[:, -1].float().argmax(-1)
        total = time.perf_counter() - t0
        return sum(layer_t), total - sum(layer_t)
    torch.set_num_threads(os.cpu_count())
    x = (torch.randn(1, ctx, H, generator=g) * 0.02).to(torch.bfloat16)
    mask = torch.ones(1, ctx, dtype=torch.long)
    step(x, mask, DynamicCache(config=cfg))                                  # warm-up
    cache = DynamicCache(config=cfg)
    layers_s, head_s = step(x, mask, cache)
    prefill_s = layers_s * lc["num_hidden_layers"] / layers_sampled + head_s
    torch.set_num_threads(threads)
    per_tok = []
    t_start = time.time()
    for i in range(tokens + 1):
        e = (torch.randn(1, 1, H, generator=g) * 0.02).to(torch.bfloat16)
        mask = torch.cat((mask, torch.ones(1, 1, dtype=torch.long)), dim=1)
        layers_s, head_s = step(e, mask, cache)
        if i > 0:  # first step is warm-up
            per_tok.append((layers_s / layers_sampled, head_s))
        if time.time() - t_start > budget_s and len(per_tok) >= 1:
            break
    return prefill_s, per_tok, ("transformers %s LlamaForCausalLM, eager attention — the reference's own decoder class "
                                "(Emu2/emu/lm.py:38; pinned 4.31.0)" % transformers.__version__)


def cpu_decode_sample(lc, vocab, layers_sampled=2, tokens=8, ctx=75, threads=None, budget_s=25.0, vc=None):
    """The reference's CPU path for the headline workload, on a bounded sample, via the oracle (oracle/emu_oracle.py):
    one real-shape EVA-CLIP block over the 1025 image tokens (x vit layers), the 75-token prompt through `layers_sampled`
    real-shape LLaMA layers (x layers / sampled), then `tokens` single-token decode steps with the KV cache + lm_head
    (per-layer time x layers).  Returns whole-job tok/s = new_tokens / (vit + prefill + new_tokens * per_token)."""
    from oracle import emu_oracle as O
    import torch.nn.functional as Fn
    global _CPU_BEST_THREADS
    if vc is None:
        vc = emu2_cfgs(False)[0] if lc["hidden_size"] > 1024 else emu2_cfgs(True)[0]
    probe = threads is None and _CPU_BEST_THREADS is None
    threads = threads or _CPU_BEST_THREADS or os.cpu_count()
    torch.set_num_threads(threads)
    H, F, nh = lc["hidden_size"], lc["intermediate_size"], lc["num_attention_heads"]
    g = torch.Generator().manual_seed(0)
    sd = _cpu_state(lc, vc, vocab, layers_sampled, g)
    with torch.no_grad():
        if probe:
            # torch's CPU bf16 matrix-vector kernels do not scale to every thread count: give the reference its best
            # setting (all cores, half, a quarter ...) from a one-layer decode probe, once per process
            best = None
            e = (torch.randn(1, 1, H, generator=g) * 0.02).to(torch.bfloat16)
            w = sd["decoder.lm.model.layers.0.mlp.gate_proj.weight"]
            cands = sorted({max(1, os.cpu_count() // d) for d in (1, 2, 4, 8, 16)}, reverse=True)
            for t in cands:
                torch.set_num_threads(t)
                Fn.linear(e, w)
                t0 = time.perf_counter()
                for _ in range(3):
                    Fn.linear(e, w)
                dt = time.perf_counter() - t0
                if best is None or dt < best[0]:
                    best = (dt, t)
            threads = _CPU_BEST_THREADS = best[1]
        # ---- ViT: one post-norm block (attention + MLP) over the image tokens, all host cores ----
        torch.set_num_threads(os.cpu_count())
        n_tok = (vc.image_size // vc.patch_size) ** 2 + 1
        W = vc.width
        xv = (torch.randn(1, n_tok, W, generator=g) * 0.5).to(torch.bfloat16)
        pre = "visual.blocks.0."
        heads = W // vc.head_width

        def vit_block(x):
            n1 = lambda t: Fn.layer_norm(t, (W,), sd[pre + "norm1.weight"], sd[pre + "norm1.bias"], 1e-6)
            n2 = lambda t: Fn.layer_norm(t, (W,), sd[pre + "norm2.weight"], sd[pre + "norm2.bias"], 1e-6)
            x = x + n1(O.vit_attention(x, sd, pre, heads))
            return x + n2(O.vit_mlp(x, sd, pre))
        vit_block(xv)
        t0 = time.perf_counter()
        vit_block(xv)
        vit_s = (time.perf_counter() - t0) * vc.layers
        # ---- LLaMA: the prompt, then single-token steps with the KV cache.  Preferably through transformers' own
        # LlamaForCausalLM — the class the reference instantiates (Emu2/emu/lm.py:38) — else through the oracle port ----
        try:
            prefill_s, per_tok, llama_src = _llama_cpu_times_hf(lc, vocab, layers_sampled, sd, ctx, tokens, threads, budget_s, g)
        except Exception as ex:  # an API drift in transformers must not take the baseline down: the port computes the same
            prefill_s, per_tok, llama_src = _llama_cpu_times_port(lc, layers_sampled, sd, ctx, tokens, threads, budget_s, g)
            llama_src += " (transformers path failed: %r)" % (ex,)
    layer_s = sum(a for a, _ in per_tok) / len(per_tok)
    head_s = sum(b for _, b in per_tok) / len(per_tok)
    tok_step_s = layer_s * lc["num_hidden_layers"] + head_s
    tok_s = NEW_TOKENS / (vit_s + prefill_s + NEW_TOKENS * tok_step_s)
    sample = ("whole job = ViT + prefill + %d decode steps, each extrapolated from a real-shape sample: 1 EVA-CLIP block "
              "(width %d, %d tokens; oracle/emu_oracle.py, port of Emu2/emu/eva_vit.py) x%d = %.1f s; LLaMA via %s: the %d-token "
              "prompt through %d LLaMA-33B layers (h=%d, ffn=%d, %d heads) x%d = %.1f s; %d timed single-token decode steps through "
              "the same layers + final norm + lm_head = %.3f s/token (decode-only %.2f tok/s); bf16; torch threads = %d of %d host "
              "cores for decode (fastest of a thread-count probe), all cores for ViT / prefill" %
              (NEW_TOKENS, W, n_tok, vc.layers, vit_s, llama_src, ctx, layers_sampled, H, F, nh,
               lc["num_hidden_layers"] // layers_sampled, prefill_s, len(per_tok), tok_step_s, 1.0 / tok_step_s, threads,
               os.cpu_count()))
    global _CPU_KIND
    _CPU_KIND = "reference" if llama_src.startswith("transformers") and "failed" not in llama_src else "port"
    return tok_s, threads, sample


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vc, lc = emu2_cfgs(args.small)
    vocab = 32272
    vals = []
    threads = os.cpu_count()
    sample = ""
    for i in range(args.warmup + args.steps):
        v, threads, sample = cpu_decode_sample(lc, vocab, layers_sampled=2, tokens=8, budget_s=20.0, vc=vc)
        if i >= args.warmup:
            vals.append(v)
    val = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "tok/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * NEW_TOKENS / val, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": val, "unit": "tok/s", "cores": threads, "kind": _CPU_KIND, "sample": sample},
        "e2e": {"value": val, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(n_gpus):
    return {"workload": "Emu2 image->text: 1x448x448 image, EVA-CLIP-4B ViT + LLaMA-33B decoder, bf16, prompt 75 "
                        "tokens (1 bos + 66 image span + 8 text), 128 new tokens greedy (EOS suppressed), batch 1",
            "global_batch": 1, "new_tokens": NEW_TOKENS,
            "parallelism": "tp%d" % n_gpus if n_gpus > 1 else "single-gpu",
            "l2_policy": "inputs larger than L2 (64.6 GB of weights streamed per token vs 126 MB L2)"}


# ------------------------------------------------------------------------------------------------
# second half of the headline metric: Emu2-Gen denoise steps/s (BASELINE.json configs[2])
# ------------------------------------------------------------------------------------------------
UNET_FLOP_PER_SAMPLE_STEP = 6.74e12  # SURVEY.md §8d: 6.74 TFLOP per sample per UNet forward at 1024x1024


def emu2_unet_json():
    """the published Emu2-Gen UNet configuration (kept in the package: emu_b200/emu2/conf.py)"""
    from emu_b200.emu2.conf import EMU2_GEN_UNET
    return dict(EMU2_GEN_UNET)


def unet_param_shapes(cfg):
    """(key, shape) of every UNet parameter, diffusers naming (mirrors emu_unet_configure's module tree)."""
    boc, lpb, cd = cfg["block_out_channels"], cfg["layers_per_block"], cfg["cross_attention_dim"]
    tl = [t if "CrossAttn" in d else 0 for t, d in zip(cfg["transformer_layers_per_block"], cfg["down_block_types"])]
    nb, temb = len(boc), boc[0] * 4
    out = []

    def lin(p, o, i, bias=True):
        out.append((p + ".weight", (o, i)))
        if bias:
            out.append((p + ".bias", (o,)))

    def cv(p, o, i, k=3):
        out.append((p + ".weight", (o, i, k, k)))
        out.append((p + ".bias", (o,)))

    def nrm(p, c):
        out.append((p + ".weight", (c,)))
        out.append((p + ".bias", (c,)))

    def resnet(p, cin, cout):
        nrm(p + "norm1", cin); cv(p + "conv1", cout, cin); lin(p + "time_emb_proj", cout, temb)
        nrm(p + "norm2", cout); cv(p + "conv2", cout, cout)
        if cin != cout:
            cv(p + "conv_shortcut", cout, cin, 1)

    def tfm(p, c, n):
        nrm(p + "norm", c); lin(p + "proj_in", c, c)
        for k in range(n):
            q = "%stransformer_blocks.%d." % (p, k)
            for a, kd in (("attn1.", c), ("attn2.", cd)):
                lin(q + a + "to_q", c, c, False); lin(q + a + "to_k", c, kd, False); lin(q + a + "to_v", c, kd, False)
                lin(q + a + "to_out.0", c, c)
            for n_ in ("norm1", "norm2", "norm3"):
                nrm(q + n_, c)
            lin(q + "ff.net.0.proj", 8 * c, c); lin(q + "ff.net.2", c, 4 * c)
        lin(p + "proj_out", c, c)

    cv("conv_in", boc[0], cfg["in_channels"])
    lin("time_embedding.linear_1", temb, boc[0]); lin("time_embedding.linear_2", temb, temb)
    lin("add_embedding.linear_1", temb, cfg["projection_class_embeddings_input_dim"]); lin("add_embedding.linear_2", temb, temb)
    cin, skip = boc[0], [boc[0]]
    for i in range(nb):
        for j in range(lpb):
            resnet("down_blocks.%d.resnets.%d." % (i, j), cin, boc[i]); cin = boc[i]
            if tl[i]:
                tfm("down_blocks.%d.attentions.%d." % (i, j), cin, tl[i])
            skip.append(cin)
        if i < nb - 1:
            cv("down_blocks.%d.downsamplers.0.conv" % i, cin, cin); skip.append(cin)
    resnet("mid_block.resnets.0.", cin, cin)
    if tl[-1]:
        tfm("mid_block.attentions.0.", cin, tl[-1])
    resnet("mid_block.resnets.1.", cin, cin)
    for i in range(nb):
        ri = nb - 1 - i
        for j in range(lpb + 1):
            resnet("up_blocks.%d.resnets.%d." % (i, j), cin + skip.pop(), boc[ri]); cin = boc[ri]
            if tl[ri]:
                tfm("up_blocks.%d.attentions.%d." % (i, j), cin, tl[ri])
        if i < nb - 1:
            cv("up_blocks.%d.upsamplers.0.conv" % i, cin, cin)
    nrm("conv_norm_out", boc[0]); cv("conv_out", cfg["out_channels"], boc[0])
    return out


def make_unet_engine(tp_rank=0, tp_size=1, uid=None, seed=0):
    """Engine holding only the Emu2-Gen UNet (random-init weights of the published topology, same seed on every rank)."""
    from emu_b200 import _lib
    from emu_b200.emu2.diffusion import unet_config_from_json
    cfg = emu2_unet_json()
    eng = _lib.Engine(_lib.EmuConfig(), tp_rank=tp_rank, tp_size=tp_size, nccl_uid=uid)
    eng.unet_configure(unet_config_from_json(cfg))   # collective over the pair when tp_size == 2 (CFG-parallel exchange)
    g = torch.Generator(device="cuda").manual_seed(seed)
    for k, shp in unet_param_shapes(cfg):
        if k.endswith(".bias"):
            t = torch.zeros(shp, device="cuda", dtype=torch.bfloat16)
        elif len(shp) == 1:
            t = torch.ones(shp, device="cuda", dtype=torch.bfloat16)
        else:
            fan = 1
            for d in shp[1:]:
                fan *= d
            t = (torch.randn(shp, generator=g, device="cuda", dtype=torch.float32) * (fan ** -0.5)).to(torch.bfloat16)
        eng.load_tensor("unet." + k, t)
        del t
    return eng, cfg


def run_denoise(steps=50, warm_loops=1, timed_loops=1, batch=1, hw=128, seed=0, profile=False, eng=None, sync=None,
                latent_seed=0):
    """50 Euler steps of the Emu2-Gen denoise loop (CFG, guidance 3, 1024x1024 -> latent 128x128) on random-init weights
    of the published UNet topology, `warm_loops` untimed loops then `timed_loops` timed ones; returns dict(steps_per_s, ms_per_step, launches_per_step, finite, sha1 of the latents,
    the latents themselves).
    `eng`: a UNet engine (possibly one half of a CFG-parallel pair); `sync`: barrier used around the timed region."""
    import hashlib
    from emu_b200 import _lib
    from emu_b200.emu2.scheduler import EulerDiscreteScheduler
    own = eng is None
    if own:
        eng, cfg = make_unet_engine(seed=seed)
    else:
        cfg = emu2_unet_json()
    g = torch.Generator(device="cuda").manual_seed(1000 + latent_seed)
    sched = EulerDiscreteScheduler()
    sched.set_timesteps(steps)
    ts, sig = sched.timesteps, sched.sigmas
    ctx = torch.randn(2 * batch, 64, cfg["cross_attention_dim"], generator=g, device="cuda").to(torch.bfloat16)
    te = ctx.float().mean(1).to(torch.bfloat16).contiguous()
    tid = torch.tensor([[1024, 1024, 0, 0, 1024, 1024]] * (2 * batch), dtype=torch.int32, device="cuda")
    lat0 = torch.randn(batch, 4, hw, hw, generator=g, device="cuda") * sched.init_noise_sigma
    lat = lat0.clone()

    def loop():
        lat.copy_(lat0)
        for i in range(steps):
            eng.denoise_step(lat, float(sig[i]), float(sig[i + 1]), float(ts[i]), 3.0, ctx, te, tid)

    for _ in range(warm_loops):
        loop()
    l0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    (sync or torch.cuda.synchronize)()
    if profile:  # ncu --profile-from-start off: capture only the timed loop (tools/ncu_unet.py)
        torch.cuda.profiler.start()
    ev0.record()
    for _ in range(timed_loops):
        loop()
    ev1.record()
    (sync or torch.cuda.synchronize)()
    if profile:
        torch.cuda.profiler.stop()
    ms = ev0.elapsed_time(ev1) / (timed_loops * steps)
    launches = (_lib.launch_count() - l0) / (timed_loops * steps)
    out = {"steps_per_s": 1000.0 / ms, "ms_per_step": ms, "launches_per_step": launches,
           "finite": bool(torch.isfinite(lat).all()),
           # correctness handle: the same seeds must give the same latents on 1 GPU and on a CFG-parallel pair (bitwise)
           "latents_sha1": hashlib.sha1(lat.cpu().numpy().tobytes()).hexdigest()[:16],
           "latents_abs_mean": float(lat.abs().mean()), "latents": lat}
    if own:
        eng.close()
    return out


# ------------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------------
def run_cuda(args):
    import torch.distributed as dist
    from emu_b200 import _lib
    from emu_b200.emu2.conf import TextDecoderCfg
    from emu_b200.emu2.emu import EmuModel
    from emu_b200.emu2 import synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    uid = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        buf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            import ctypes
            raw = ctypes.create_string_buffer(128)
            _lib.check(_lib.load().emu_nccl_unique_id(raw))
            buf.copy_(torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        uid = bytes(buf.cpu().numpy().tobytes())

    vc, lc = emu2_cfgs(args.small)
    vocab = synthetic.VOCAB_EMU2
    n_query = vc.n_query
    prompt_len = 2 + n_query + 1 + N_TEXT
    model = EmuModel(vc, TextDecoderCfg(), tokenizer=synthetic.SyntheticTokenizer(vocab), llama_config=lc,
                     max_batch=5 if (world == 1 and not args.no_beam) else 1,  # 5 cache rows only for the 5-beam secondary
                     max_seq=prompt_len + NEW_TOKENS + 8, tp_rank=rank, tp_size=world, nccl_uid=uid)
    synthetic.load_random_weights(model, vc, lc, vocab, seed=0)

    g = torch.Generator().manual_seed(1234)
    image_host = torch.randn(1, 3, vc.image_size, vc.image_size, generator=g).to(torch.bfloat16).pin_memory()
    ids_host, mask_host = synthetic.image_prompt_ids(n_query=n_query, n_text=N_TEXT)
    ids_host, mask_host = ids_host.pin_memory(), mask_host.pin_memory()
    image_dev, ids_dev, mask_dev = image_host.cuda(), ids_host.cuda(), mask_host.cuda()

    def one_step(resident):
        if resident:
            toks = model.generate_from_ids(ids_dev, mask_dev, image=image_dev, num_beams=1, max_new_tokens=NEW_TOKENS,
                                           min_len=NEW_TOKENS, check_every=0)
            return toks
        img = image_host.to("cuda", non_blocking=True)
        ids = ids_host.to("cuda", non_blocking=True)
        msk = mask_host.to("cuda", non_blocking=True)
        toks = model.generate_from_ids(ids, msk, image=img, num_beams=1, max_new_tokens=NEW_TOKENS, min_len=NEW_TOKENS,
                                       check_every=0)
        return toks.cpu()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(resident, steps):
        return timed_fn(lambda: one_step(resident), steps)

    def timed_fn(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            toks = fn()
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, toks

    for _ in range(args.warmup):
        one_step(True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    ms, toks = timed(True, args.steps)
    launches = _lib.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else {}
    assert toks.shape[1] == NEW_TOKENS, toks.shape
    outputs = {"tokens": toks}
    value = args.steps * NEW_TOKENS / (ms / 1000.0)

    # end to end through the public API with host buffers
    one_step(False)
    ms_e2e, _ = timed(False, args.steps)
    e2e = args.steps * NEW_TOKENS / (ms_e2e / 1000.0)

    # correctness handle of the timed run (VERDICT r01): the 128 greedy ids, hashed, so that the N = 1/2/4/8 lines of a scaling
    # run can be compared; every tensor-parallel rank must hold the same ids (fixed-order reductions)
    import hashlib
    tok_cpu = toks.to(torch.int64).cpu().contiguous()
    tokens_sha1 = hashlib.sha1(tok_cpu.numpy().tobytes()).hexdigest()[:16]
    ranks_agree = True
    if world > 1:
        mine = torch.tensor([int(tokens_sha1, 16) >> 1], dtype=torch.int64, device="cuda")
        allh = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allh, mine)
        ranks_agree = all(int(h.item()) == int(mine.item()) for h in allh)

    # ViT and prefill times of the same request (SURVEY.md §8d: reported separately from decode tok/s)
    eng = model.engine

    def ev_ms(fn, reps=3):
        fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            out = fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps, out
    vit_ms, e = ev_ms(lambda: model.encode_image(image_dev))
    emb = eng.llm_embed(ids_dev)
    emb[ids_dev == 32003] = model._project_up(e.reshape(-1, e.shape[-1]))

    def prefill():
        eng.llm_reset()
        return eng.llm_prefill(emb, mask_dev, hf_positions=True, want_logits=True)
    prefill_ms, _ = ev_ms(prefill)

    # decode-step timing for the roofline: events around each CUDA-graphed decode step of one more generate
    eng.llm_reset()
    _, logits = eng.llm_prefill(emb, mask_dev, hf_positions=True, want_logits=True)
    ping = [logits.argmax(-1).to(torch.int32), torch.empty(1, dtype=torch.int32, device="cuda")]
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(NEW_TOKENS)]
    torch.cuda.synchronize()
    evs[0].record()
    for s in range(1, NEW_TOKENS):
        eng.llm_decode(token_ids=ping[(s - 1) & 1], next_ids=ping[s & 1], ban_id=2, B=1)
        evs[s].record()
    torch.cuda.synchronize()
    step_ms = sorted(evs[s - 1].elapsed_time(evs[s]) for s in range(1, NEW_TOKENS))
    step_ms_avg = sum(step_ms) / len(step_ms)

    # secondary (SURVEY.md §8d): the reference's default decoding — 5 beams, length_penalty -1 — same prompt and length
    beam5 = None
    if not args.no_beam and world == 1:
        try:
            def beam_gen():
                return model.generate_from_ids(ids_dev, mask_dev, image=image_dev, num_beams=5, max_new_tokens=NEW_TOKENS,
                                               min_len=NEW_TOKENS, length_penalty=-1)
            beam_gen()
            ms_b, tb = timed_fn(beam_gen, 1)
            beam5 = {"metric": "emu2_img2text_beam5_tok_per_s", "value": tb.shape[1] / (ms_b / 1000.0), "unit": "tok/s",
                     "new_tokens": int(tb.shape[1]), "ms": ms_b,
                     "tokens_sha1": hashlib.sha1(tb.to(torch.int64).cpu().numpy().tobytes()).hexdigest()[:16],
                     "config": "num_beams=5, length_penalty=-1 (reference default), batch 1 -> 5 cache rows, "
                               "device-side emu_beam_topk + emu_beam_step per step (no host synchronisation in the loop)"}
        except Exception as ex:
            beam5 = {"metric": "emu2_img2text_beam5_tok_per_s", "value": None, "error": repr(ex)}
    ctx_avg = prompt_len + NEW_TOKENS / 2.0
    alg_bytes = (llm_bytes_per_token(lc, vocab) + kv_bytes_per_ctx_token(lc) * ctx_avg) / world
    peak, peak_src = measured_peaks()
    achieved = alg_bytes / (step_ms_avg / 1000.0) / 1e9

    # ---- second half of the headline metric: Emu2-Gen denoise steps/s at this GPU count ----
    # N = 1: batch 1 + CFG on one GPU.  N = 2: CFG-parallel pair (cond on rank 0, uncond on rank 1, noise predictions swapped
    # over NVLink inside the CFG+Euler kernel).  N = 4 / 8: N/2 such pairs, each denoising its own image (UNet tensor
    # parallelism at batch 1 does not pay: SURVEY.md §8e) — value = images x steps / s over the whole job.
    denoise = None
    if not args.small and not args.no_denoise:
        try:
            del model
            torch.cuda.empty_cache()
            bf16_peak = 1739.4
            try:
                bf16_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
            except Exception:
                pass
            if world == 1:
                r = run_denoise(warm_loops=args.warmup, timed_loops=args.steps)
                images, layout = 1, "1 GPU: UNet batch 2 (cond + uncond)"
            else:
                import ctypes
                pair, prank = rank // 2, rank % 2
                mine = torch.zeros(128, dtype=torch.uint8, device="cuda")
                if prank == 0:
                    raw = ctypes.create_string_buffer(128)
                    _lib.check(_lib.load().emu_nccl_unique_id(raw))
                    mine.copy_(torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8))
                alls = [torch.zeros_like(mine) for _ in range(world)]
                dist.all_gather(alls, mine)
                puid = bytes(alls[pair * 2].cpu().numpy().tobytes())   # the id made by the even rank of my pair
                ueng, _ = make_unet_engine(tp_rank=prank, tp_size=2, uid=puid)
                r = run_denoise(eng=ueng, sync=barrier, latent_seed=pair, warm_loops=args.warmup, timed_loops=args.steps)
                t = torch.tensor([r["ms_per_step"]], device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                r["ms_per_step"] = float(t.item())
                # both ranks of a pair must hold bitwise identical latents
                hv = torch.tensor([int(r["latents_sha1"], 16) >> 1], dtype=torch.int64, device="cuda")
                hs = [torch.zeros_like(hv) for _ in range(world)]
                dist.all_gather(hs, hv)
                r["pair_latents_identical"] = all(int(hs[2 * q].item()) == int(hs[2 * q + 1].item()) for q in range(world // 2))
                r["latents_sha1_per_pair"] = ["%016x" % (int(hs[2 * q].item()) << 1) for q in range(world // 2)]
                images, layout = world // 2, "%d CFG-parallel pair(s): cond on even ranks, uncond on odd ranks, one image per pair" % (world // 2)
                ueng.close()
            outputs["denoise_latents"] = r["latents"]
            sps = images * 1000.0 / r["ms_per_step"]
            ach = images * 2 * UNET_FLOP_PER_SAMPLE_STEP / (r["ms_per_step"] / 1000.0) / 1e12
            denoise = {"metric": "emu2gen_denoise_steps_per_s", "value": sps, "unit": "steps/s", "ms_per_step": r["ms_per_step"],
                       "images_in_flight": images, "scaling": "strong 1->2 (one image), weak beyond (one image per pair)",
                       "config": "SDXL-topology UNet 2.53B, 1024x1024 (latent 128x128), batch 1 + CFG per image, 50 Euler "
                                 "steps, guidance 3, ctx [2,64,1792], bf16, CUDA-graphed fused step; " + layout,
                       "timed_loops": args.steps, "warmup_loops": args.warmup,   # loops of 50 steps, from --steps / --warmup
                       "gpu_launches_per_step": r["launches_per_step"], "finite": r["finite"],
                       "latents_sha1": r["latents_sha1"], "latents_abs_mean": r["latents_abs_mean"],
                       "pair_latents_identical": r.get("pair_latents_identical"),
                       "latents_sha1_per_pair": r.get("latents_sha1_per_pair"),
                       "roofline": {"bound": "tensor", "achieved": ach, "peak": bf16_peak * world, "unit": "TFLOP/s",
                                    "frac": ach / (bf16_peak * world), "flops_per_step": images * 2 * UNET_FLOP_PER_SAMPLE_STEP,
                                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained x n_gpus"}}
        except Exception as ex:
            denoise = {"metric": "emu2gen_denoise_steps_per_s", "value": None, "error": repr(ex)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            v, threads, sample = cpu_decode_sample(lc, vocab, layers_sampled=2, tokens=8, budget_s=25.0, vc=vc)
            cpu = {"value": v, "unit": "tok/s", "cores": threads, "kind": _CPU_KIND, "sample": sample}
        except Exception as ex:  # the CPU baseline must never take the GPU result down with it
            cpu = {"value": None, "unit": "tok/s", "cores": os.cpu_count(), "kind": "port", "sample": "failed: %r" % ex}

    traffic_ratio, traffic_src = ncu_traffic()
    line = {
        "metric": METRIC, "value": value, "unit": "tok/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "config": workload_config(world),
        "e2e": {"value": e2e, "unit": "tok/s", "h2d_bytes_per_step": int(image_host.numel() * 2 + ids_host.numel() * 16),
                "d2h_bytes_per_step": int(NEW_TOKENS * 8)},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "gemv_tma_kernel (the weight-streaming launches of one decode step; "
                     ">95% of the CUDA-graphed step)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "peak_source": peak_src,
                     # ncu --set full on the gate/up launch (profiles/r01_ncu_full_gemv_tma_gateup.txt): dram read
                     # 477.3 MB + write 6.5 MB for 477.1 MB of weights -> x1.014 of the algorithmic bytes, per step here
                     "traffic": (alg_bytes * traffic_ratio) if traffic_ratio else None,
                     "traffic_source": ("ncu dram__bytes_read+write / algorithmic bytes of the gate_up launch (x%.3f, %s), "
                                        "scaled to the step" % (traffic_ratio, traffic_src)) if traffic_ratio else None,
                     "decode_step_ms": step_ms_avg, "decode_step_ms_p50": step_ms[len(step_ms) // 2],
                     "algorithmic_bytes_per_step": alg_bytes},
        "cpu_baseline": cpu,
        "tokens_sha1": tokens_sha1, "tokens_head": [int(v) for v in tok_cpu[0, :8]], "tokens_identical_across_ranks": ranks_agree,
        "vit_ms": vit_ms, "prefill_ms": prefill_ms,
        "denoise": denoise,
        "beam5": beam5,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# BASELINE configs[3]: interleaved 8-shot prompts (seq ~4k), batch 4, the reference's default 5-beam decoding, LLaMA-33B tensor
# parallel over the box (Emu2/README.md:221-246, Emu2/emu/emu.py:189-229)
# ------------------------------------------------------------------------------------------------
def c4_prompt_ids(n_query=64, shots=8, n_text=440, batch=4, seed=0):
    from emu_b200.emu2.synthetic import IDS
    g = torch.Generator().manual_seed(seed)
    span = torch.tensor([IDS["[IMG]"]] + [IDS["<image>"]] * n_query + [IDS["[/IMG]"]])
    rows = []
    for _ in range(batch):
        parts = [torch.tensor([IDS["bos"]])]
        for _ in range(shots):
            parts += [span, torch.randint(100, 31000, (n_text,), generator=g)]
        rows.append(torch.cat(parts))
    ids = torch.stack(rows)
    return ids, torch.ones_like(ids)


def run_c4(args):
    import hashlib
    import torch.distributed as dist
    from emu_b200 import _lib
    from emu_b200.emu2.conf import TextDecoderCfg
    from emu_b200.emu2.emu import EmuModel
    from emu_b200.emu2 import synthetic
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    uid = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        buf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            import ctypes
            raw = ctypes.create_string_buffer(128)
            _lib.check(_lib.load().emu_nccl_unique_id(raw))
            buf.copy_(torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        uid = bytes(buf.cpu().numpy().tobytes())
    vc, lc = emu2_cfgs(args.small)
    vocab = synthetic.VOCAB_EMU2
    shots, n_text, batch, beams = (8, 440, 4, 5) if not args.small else (2, 6, 2, 3)
    ids_host, mask_host = c4_prompt_ids(vc.n_query, shots, n_text, batch)
    prompt_len = ids_host.shape[1]
    new_tokens = NEW_TOKENS if not args.small else 8
    model = EmuModel(vc, TextDecoderCfg(), tokenizer=synthetic.SyntheticTokenizer(vocab), llama_config=lc,
                     max_batch=batch * beams, max_seq=prompt_len + new_tokens + 8, tp_rank=rank, tp_size=world, nccl_uid=uid)
    synthetic.load_random_weights(model, vc, lc, vocab, seed=0)
    g = torch.Generator().manual_seed(4321)
    images_host = torch.randn(batch * shots, 3, vc.image_size, vc.image_size, generator=g).to(torch.bfloat16).pin_memory()
    ids_host, mask_host = ids_host.pin_memory(), mask_host.pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step():
        img = images_host.to("cuda", non_blocking=True)
        ids = ids_host.to("cuda", non_blocking=True)
        msk = mask_host.to("cuda", non_blocking=True)
        return model.generate_from_ids(ids, msk, image=img, num_beams=beams, max_new_tokens=new_tokens, min_len=new_tokens,
                                       length_penalty=-1).cpu()
    for _ in range(args.warmup):
        one_step()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = _lib.launch_count()
    ev0.record()
    for _ in range(args.steps):
        toks = one_step()
    ev1.record()
    barrier()
    launches = _lib.launch_count() - l0
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    # the pieces, timed separately on the same inputs
    img, ids, msk = images_host.cuda(), ids_host.cuda(), mask_host.cuda()

    def ev_ms(fn):
        fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        out = fn()
        b.record()
        barrier()
        return a.elapsed_time(b), out
    vit_ms, e = ev_ms(lambda: model.encode_image(img))
    emb = model.engine.llm_embed(ids)
    emb[ids == 32003] = model._project_up(e.reshape(-1, e.shape[-1]))

    def prefill():
        model.engine.llm_reset()
        return model.engine.llm_prefill(emb, msk, hf_positions=True, want_logits=True)
    prefill_ms, _ = ev_ms(prefill)
    decode_ms = ms / args.steps - vit_ms - prefill_ms
    step_ms = decode_ms / max(1, new_tokens - 1)
    H, L = lc["hidden_size"], lc["num_hidden_layers"]
    tokens = batch * prompt_len
    prefill_flops = 2.0 * (llm_bytes_per_token(lc, vocab) / 2) * tokens + 4.0 * L * batch * prompt_len * prompt_len / 2 * H
    kv_bytes = kv_bytes_per_ctx_token(lc) * (prompt_len + new_tokens / 2.0) * batch * beams
    alg_bytes = (llm_bytes_per_token(lc, vocab) + kv_bytes) / world
    peak, peak_src = measured_peaks()
    bf16_peak = 1480.4
    try:
        bf16_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
    except Exception:
        pass
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"tokens": toks})
        emit({
            "metric": "emu2_c4_interleaved_tok_per_s", "value": args.steps * batch * new_tokens / (ms / 1000.0), "unit": "tok/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "Emu2 interleaved in-context (BASELINE configs[3]): %d prompts x %d shots of (66-token image "
                                   "span + %d text tokens) = %d prompt tokens each, %d images through the ViT (data-parallel over "
                                   "ranks), LLaMA-33B, %d beams (reference default, length_penalty -1) -> %d cache rows, %d new "
                                   "tokens per prompt" % (batch, shots, n_text, prompt_len, batch * shots, beams, batch * beams,
                                                          new_tokens),
                       "parallelism": "tp%d" % world, "global_batch": batch},
            "e2e": {"value": args.steps * batch * new_tokens / (ms / 1000.0), "unit": "tok/s",
                    "h2d_bytes_per_step": int(images_host.numel() * 2 + ids_host.numel() * 16), "d2h_bytes_per_step": int(batch * new_tokens * 8)},
            "gpu_launches": int(launches),
            "vit_ms": vit_ms, "prefill_ms": prefill_ms, "decode_ms": decode_ms, "decode_step_ms": step_ms,
            "tokens_sha1": hashlib.sha1(toks.to(torch.int64).numpy().tobytes()).hexdigest()[:16],
            "roofline": {"bound": "hbm", "kernel": "wide decode step: gemm_skinny_kernel (tcgen05, weights as the 128-row operand, %d cache rows as N) + split-KV attn_decode_kernel through the beam row table" % (batch * beams),
                         "achieved": alg_bytes / (step_ms / 1000.0) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg_bytes / (step_ms / 1000.0) / 1e9 / peak, "peak_source": peak_src,
                         "algorithmic_bytes_per_step_per_gpu": alg_bytes, "traffic": None},
            "prefill_roofline": {"bound": "tensor", "achieved": prefill_flops / world / (prefill_ms / 1000.0) / 1e12, "peak": bf16_peak,
                                 "unit": "TFLOP/s per GPU", "frac": prefill_flops / world / (prefill_ms / 1000.0) / 1e12 / bf16_peak,
                                 "flops": prefill_flops},
        })
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# BASELINE configs[4]: batched text->image, 32 prompts, 50 steps, 1024x1024, UNet over the box.  Independent samples shard
# trivially (SURVEY.md §8e): every rank keeps the whole UNet (5 GB) and denoises 32 / N prompts with its cond / uncond pairs
# together (CFG combine stays local) — no collective in the loop, final latents stay where the VAE decode would run.
# ------------------------------------------------------------------------------------------------
def run_c5(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    prompts = 32
    per = (prompts + world - 1) // world
    mine = max(0, min(per, prompts - rank * per))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    eng, _ = make_unet_engine()
    r = run_denoise(eng=eng, sync=barrier, batch=max(mine, 1), latent_seed=rank, warm_loops=args.warmup,
                    timed_loops=args.steps)
    eng.close()
    ms_loop = r["ms_per_step"]
    if world > 1:
        t = torch.tensor([ms_loop], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_loop = float(t.item())
    bf16_peak = 1480.4
    try:
        bf16_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
    except Exception:
        pass
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"denoise_latents": r["latents"]})
        ach = prompts * 2 * UNET_FLOP_PER_SAMPLE_STEP / (ms_loop / 1000.0) / 1e12
        emit({"metric": "emu2gen_c5_image_steps_per_s", "value": prompts * 1000.0 / ms_loop, "unit": "image-steps/s",
              "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_loop, "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
              "config": {"workload": "Emu2-Gen batched text->image (BASELINE configs[4]): 32 prompts, 50 Euler steps, 1024x1024, "
                                     "guidance 3 (UNet batch 64), %d prompts per GPU with their cond/uncond pairs together, "
                                     "weights replicated, no collective in the loop" % per, "parallelism": "dp%d" % world,
                         "global_batch": prompts},
              "e2e": {"value": prompts * 1000.0 / ms_loop, "unit": "image-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
              "gpu_launches": int(r["launches_per_step"] * 50), "time_for_50_steps_s": ms_loop * 50 / 1000.0,
              "latents_sha1_rank0": r["latents_sha1"], "finite": r["finite"],
              "roofline": {"bound": "tensor", "achieved": ach, "peak": bf16_peak * world, "unit": "TFLOP/s", "frac": ach / (bf16_peak * world),
                           "traffic": None}})
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def quiet_stdout():
    """Route fd 1 to stderr for the run (NCCL and other native libraries print banners to stdout); the one JSON line
    goes to the real stdout through emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3,
                    help="timed steps: generate calls (c2, c4) and 50-step denoise loops (the denoise half of c2, c5)")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps of the same kinds before the timed ones")
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--small", action="store_true", help="tiny plumbing config (debug only; never a bench number)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-denoise", action="store_true", help="skip the Emu2-Gen denoise-loop measurement")
    ap.add_argument("--no-beam", action="store_true", help="skip the secondary 5-beam measurement")
    ap.add_argument("--config", default="c2", choices=["c2", "c4", "c5"],
                    help="c2 = BASELINE configs[1] (the headline, default); c4 = configs[3]: 8-shot interleaved prompts "
                         "(seq ~4k), batch 4, 5 beams, LLaMA-33B tensor parallel over --gpus (needs >= 2 GPUs for the KV cache); "
                         "c5 = configs[4]: 32 prompts x 50 denoise steps at 1024x1024, the prompt batch sharded over --gpus")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (greedy token ids; the final latents of "
                         "the denoise loop) as DIR/<name>.npy, float32 / float64, to compare two builds on the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA arm: the reference arm only times a sample of the work")
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback (use --impl reference for the CPU arm)")
    if args.config == "c4":
        run_c4(args)
        return
    if args.config == "c5":
        run_c5(args)
        return
    run_cuda(args)


if __name__ == "__main__":
    main()
