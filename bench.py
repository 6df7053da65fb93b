"""bench.py -- the driver's benchmark contract for the video-conversation hot path.

    python bench.py --gpus N --steps K --warmup W [--impl vcl|reference|library]
                    [--config 2|3|4|5] [--clips B] [--model 7b|13b] [--frames 32,64,100]
                    [--dump-outputs DIR]

Configurations (numbering of SURVEY.md 8d; BASELINE.json `configs` is 0-based, so config k = configs[k-1]):
  2  (default, the configuration the metric is quoted on) 1 clip per GPU: 100 synthetic 224x224
     frames -> CLIP ViT-L/14 (23 layers) -> spatio-temporal pool -> mm_projector + splice into a
     448-token prompt -> Vicuna-7B prefill -> exactly 32 greedy tokens (EOS ignored)
  3  the same with 16 clips per GPU (batched prefill / decode)
  4  Vicuna-13B, 4 clips per GPU (32 clips over 8 GPUs)
  5  CLIP-only extraction sweep: a job of 1000 clips at each of T = 32 / 64 / 100 frames, clips dealt
     round-robin to the GPUs; one step = one clip at every T on every GPU
Random-init bf16 weights of the named architecture, synthetic frames (no checkpoints / datasets are
reachable offline). With N GPUs every rank runs its own clips (clips are independent: weak scaling)
and the step ends with one NCCL all_gather of the token ids (config 5: of per-clip checksums) --
the only collective on the path.

Printed JSON (rank 0, one line):
  value / ms_per_step  device-resident: frames, ids already in HBM when the timed region starts; the
                       engine is driven through the C ABI directly
  e2e                  the same metric through the REFERENCE-FACING API with HOST (pinned) buffers:
                       vision_tower(frames).hidden_states[-2][:, 1:] -> get_spatio_temporal_features_torch
                       -> model.generate(...) (video_chatgpt/inference.py:86-112), uint8 frames + ids copied
                       H2D and the token ids copied D2H inside the timed region
  roofline             the dominant stage at 1 clip/GPU is the weight-streaming decode loop (HBM-bound):
                       achieved = algorithmic bytes of the 31 decode steps / their device time, taken
                       with CUDA events inside the timed region, against MEASURED_PEAKS.json
  stages               per-stage device time and achieved TFLOP/s (ViT / prefill: tensor-bound)
  cpu_baseline         the oracle (a port of the reference's path) timed on the host cores on ONE bounded
                       sample, extrapolated to the full workload (sample stated)
  library_baseline     the same oracle in bf16 on THIS GPU through stock PyTorch kernels (eager attention,
                       as the reference's HF code runs it, and SDPA): what the reference's Python would
                       cost on the box (SURVEY.md 2.3); 1 warm-up + 1 timed clip
`--impl reference` times the CPU path as the arm of its own (rank 0 only; one bounded sample whatever
--steps says); `--impl library` prints the library baseline alone.

`--dump-outputs DIR` (--impl vcl) writes what the last timed device-resident step returned, on rank 0, as
DIR/<name>.npy in float32: `tokens` [clips, 32] (all ranks' clips with N GPUs) and `video_features`
[clips, 356, 1024] (configs 2-4), or `video_features_T<t>` [356, 1024] per frame count (config 5). Weights
and inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "video-llava_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

T_FRAMES, N_NEW, S_PROMPT = 100, 32, 448
MODELS = {"7b": dict(hidden=4096, inter=11008, heads=32, layers=32),
          "13b": dict(hidden=5120, inter=13824, heads=40, layers=40)}
CONFIGS = {2: dict(model="7b", clips=1, label="configs[1]: single clip, 100 frames -> Vicuna-7B greedy 32-token answer"),
           3: dict(model="7b", clips=16, label="configs[2]: batch=16 clips x 100 frames, Vicuna-7B bf16, one GPU"),
           4: dict(model="13b", clips=4, label="configs[3]: Vicuna-13B, 100-frame clips, 4 clips per GPU (batch 32 over 8 GPUs)"),
           5: dict(model="7b", clips=1, label="configs[4]: CLIP-only throughput sweep, 1000 clips x {32,64,100} frames")}
METRIC = "videos/sec (100-frame CLIP encode + 7B 32-tok decode)"
SWEEP_CLIPS = 1000
DUMP_BYTES = 60 * 10 ** 6          # --dump-outputs: array data in all, under 64 MB with the .npy headers


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1400.0, "fallback"


# ---------------------------------------------------------------------------------------------
# algorithmic work (SURVEY.md section 8d)
# ---------------------------------------------------------------------------------------------
VIT_FLOPS_PER_FRAME = 23 * (2 * 257 * 1024 * 3072 + 2 * 257 * 1024 * 1024 + 4 * 257 * 257 * 1024 +
                            4 * 257 * 1024 * 4096) + 2 * 256 * 588 * 1024


def work(model):
    m = MODELS[model]
    D, F, L, V = m["hidden"], m["inter"], m["layers"], 32003
    body = L * (4 * D * D + 3 * D * F)
    prefill = 2 * S_PROMPT * body + L * 2 * S_PROMPT * S_PROMPT * D + 2 * 356 * 1024 * D + 2 * D * V
    weights_step = (body + V * D) * 2                      # bytes streamed per decode step
    kv_per_tok = L * 2 * D * 2                             # bytes per cached token per clip
    return dict(vit_flops=VIT_FLOPS_PER_FRAME * T_FRAMES, prefill_flops=prefill, weights_step=weights_step,
                kv_per_tok=kv_per_tok)


def workload_config(cfg_id, model, B, world):
    """The `config` object of the JSON line -- the same for every --impl, so the arms are comparable."""
    w = work(model)
    if cfg_id == 5:
        return {"workload": f"{CONFIGS[5]['label']}; per clip: T synthetic 224x224 frames -> CLIP ViT-L/14 (23 layers) -> "
                            f"spatio-temporal pool -> [356,1024] fp16",
                "job": f"{SWEEP_CLIPS} clips per T, dealt round-robin to the GPUs; value = clips/s summed over the three T",
                "parallelism": f"dp{world} (clips sharded, one all_gather of per-clip checksums)",
                "weights": "random-init bf16 (seed 0)",
                "l2": "no flush: every clip streams its own frames and activations (0.7 GB per 100-frame clip) through "
                      "the 126 MB L2"}
    return {"workload": f"{CONFIGS[cfg_id]['label']}; per clip: {T_FRAMES} frames 224x224 -> CLIP ViT-L/14 (23 layers) -> pool -> "
                        f"projector -> Vicuna-{model.upper()} prefill S={S_PROMPT} -> {N_NEW} greedy tokens",
            "clips_per_gpu": B, "parallelism": f"dp{world} (clips sharded, one all_gather of token ids)",
            "weights": "random-init bf16 (seed 0)",
            "l2": "no flush: every step streams inputs+weights far larger than L2 "
                  f"({w['weights_step'] / 1e9:.1f} GB of weights per decode step vs 126 MB)"}


def dump_outputs(path, arrays):
    """Write {name: tensor} as path/<name>.npy in float32 (token ids below 2^24 stay exact). Smallest first,
    an array larger than its share of what is left of DUMP_BYTES keeps a fixed, seeded subset of its
    leading-axis rows, so a larger --clips still gives the same rows on every run."""
    os.makedirs(path, exist_ok=True)
    left = DUMP_BYTES
    for i, (name, t) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].numel())):
        a = t.float().cpu().numpy()
        share = left // (len(arrays) - i)
        if a.nbytes > share:
            keep = max(1, share * len(a) // a.nbytes)
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)
        left -= a.nbytes


def metric_name(cfg_id, model):
    if cfg_id == 5:
        return "videos/sec (CLIP ViT-L/14 encode + pool, mean over T = 32/64/100 frames)"
    return METRIC if model == "7b" else METRIC.replace("7B", "13B")


# ---------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi in the background during the timed region)
# ---------------------------------------------------------------------------------------------
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle (port of the reference path) on ONE bounded sample
# ---------------------------------------------------------------------------------------------
def host_cores():
    """Cores this process may really use: the affinity mask, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


def pick_threads():
    """The intra-op thread count at which a prefill-shaped fp32 GEMM runs fastest on this host
    (oversubscribing a 128-thread box is slower than using 32-64 of its threads)."""
    avail = host_cores()
    cands = sorted({c for c in (8, 16, 32, 64, 96, avail) if c <= avail} | {avail})
    a, b = torch.randn(448, 4096), torch.randn(4096, 11008)
    best, best_t, probe = cands[-1], None, {}
    for c in cands:
        torch.set_num_threads(c)
        a @ b
        t0 = time.perf_counter()
        for _ in range(3):
            a @ b
        t = (time.perf_counter() - t0) / 3
        probe[c] = round(2 * 448 * 4096 * 11008 / t / 1e9, 1)
        if best_t is None or t < best_t * 0.97:     # prefer fewer threads unless more is clearly faster
            best, best_t = c, t
    torch.set_num_threads(best)
    return best, avail, probe


_CPU_WEIGHTS = {}
CPU_BUDGET_S = 110.0


def cpu_sample(model="7b", budget_s=CPU_BUDGET_S):
    """Times oracle/vcl_oracle.py on the host in fp32 (the fastest CPU arithmetic when there is no AMX;
    fixed, so runs are comparable): the reference's CLIP as it executes it (all 24 layers) on a few
    frames, the reference pool on a full [100,256,1024] tensor, and a few full-width LLaMA layers for
    a 448-token prefill (logits for all positions, as the reference computes them) plus cached decode
    steps; extrapolated linearly in frames / layers / steps (the layers are identical, the CLIP cost is
    linear in frames). The sample grows until about budget_s/2 of timed work is reached and never
    exceeds budget_s: ONE bounded sample, whatever --steps says."""
    from oracle import vcl_oracle as O
    t_all = time.perf_counter()
    threads, avail, probe = pick_threads()
    dtype = torch.float32
    m = MODELS[model]
    L = m["layers"]
    ccfg = O.ClipCfg()
    l_layers = 2
    lcfg = O.LlmCfg(hidden=m["hidden"], inter=m["inter"], heads=m["heads"], layers=l_layers)
    left = lambda: budget_s - (time.perf_counter() - t_all)
    with torch.no_grad():
        key = (model, l_layers)
        if key not in _CPU_WEIGHTS:            # random-init weights are built once per process
            _CPU_WEIGHTS[key] = (O.random_clip_state(ccfg, seed=0, n_layers=24), O.random_llm_state(lcfg, seed=0))
        csd, lsd = _CPU_WEIGHTS[key]
        px = O.preprocess_frames(O.make_frames(0, 16))
        t0 = time.perf_counter(); O.clip_hidden_states(csd, ccfg, px[:1], 24); t1 = time.perf_counter() - t0   # warm-up + estimate
        t_frames = int(max(1, min(16, 0.25 * left() / max(t1, 1e-3))))
        t0 = time.perf_counter(); O.clip_hidden_states(csd, ccfg, px[:t_frames], 24); t_clip = time.perf_counter() - t0
        feats = torch.randn(100, 256, 1024)
        t0 = time.perf_counter(); pooled = O.st_pool_torch(feats); t_pool = time.perf_counter() - t0
        ids = O.make_prompt_ids(lcfg, 356, seed=1)
        vf = pooled[None].to(dtype)
        t0 = time.perf_counter()
        logits, _, past = O.llm_forward(lsd, lcfg, ids, vf, all_logits=True)
        t_pre = time.perf_counter() - t0
        if left() > 4 * t_pre + 20:            # second pass: caches / thread pool are warm now
            t0 = time.perf_counter()
            logits, _, past = O.llm_forward(lsd, lcfg, ids, vf, all_logits=True)
            t_pre = min(t_pre, time.perf_counter() - t0)
        lcfg0 = O.LlmCfg(hidden=m["hidden"], inter=m["inter"], heads=m["heads"], layers=0)
        t0 = time.perf_counter()
        O.llm_forward(lsd, lcfg0, ids, vf, all_logits=True)               # embed + splice + norm + lm_head only
        t_pre_fixed = time.perf_counter() - t0
        tok = logits[:, -1].argmax(-1)
        dec_steps, t_dec = 0, 0.0
        t0 = time.perf_counter()
        while dec_steps < 8 and (dec_steps < 2 or left() > 15):
            logits, _, past = O.llm_forward(lsd, lcfg, tok[:, None], vf, past)
            tok = logits[:, -1].argmax(-1)
            dec_steps += 1
        t_dec = (time.perf_counter() - t0) / dec_steps
        t0 = time.perf_counter()
        O.llm_forward(lsd, lcfg0, tok[:, None], vf, None)                 # embed + norm + lm_head of one token
        t_dec_fixed = time.perf_counter() - t0
    per_layer_pre = max(t_pre - t_pre_fixed, 0.0) / l_layers
    per_layer_dec = max(t_dec - t_dec_fixed, 0.0) / l_layers
    clip_full = t_clip * T_FRAMES / t_frames
    pre_full = t_pre_fixed + per_layer_pre * L
    dec_full = (t_dec_fixed + per_layer_dec * L) * (N_NEW - 1)
    total = clip_full + t_pool + pre_full + dec_full
    return {
        "value": 1.0 / total, "unit": "videos/s", "cores": threads, "cores_available": avail, "kind": "port",
        "dtype": "f32", "thread_probe_gflops": probe,
        "sample": (f"oracle (port of the reference path) in float32 on {threads} of {avail} usable host threads: "
                   f"24-layer CLIP on {t_frames} frames ({t_clip:.2f}s), pool [100,256,1024] ({t_pool * 1e3:.1f}ms), "
                   f"{l_layers} of {L} {model} layers: 448-token prefill with all-position logits ({t_pre:.2f}s), "
                   f"{dec_steps} cached decode steps ({t_dec:.3f}s each); scaled linearly to 100 frames, {L} layers, "
                   f"{N_NEW - 1} steps -> {total:.1f}s per clip (CLIP {clip_full:.1f} + prefill {pre_full:.1f} + decode {dec_full:.1f})"),
        "seconds_sampled": time.perf_counter() - t_all,
    }


# ---------------------------------------------------------------------------------------------
# weights / inputs
# ---------------------------------------------------------------------------------------------
def device_weights(model, dev):
    """Random-init bf16 weights of the named architecture, generated on the device (seed 0)."""
    m = MODELS[model]
    D, F, L, V = m["hidden"], m["inter"], m["layers"], 32003
    g = torch.Generator(device=dev).manual_seed(0)
    rn = lambda *s, std: (torch.randn(*s, device=dev, dtype=torch.float32, generator=g) * std).to(torch.bfloat16)
    big = lambda r, c, std: torch.empty(r, c, device=dev, dtype=torch.bfloat16).normal_(0.0, std, generator=g)
    C, CF, P = 1024, 4096, 256
    p = "vision_model."
    clip = {p + "embeddings.class_embedding": rn(C, std=C ** -0.5),
            p + "embeddings.patch_embedding.weight": rn(C, 3, 14, 14, std=0.02),
            p + "embeddings.position_embedding.weight": rn(P + 1, C, std=0.02),
            p + "pre_layrnorm.weight": 1 + rn(C, std=0.05), p + "pre_layrnorm.bias": rn(C, std=0.02)}
    for l in range(23):
        lp = f"{p}encoder.layers.{l}."
        for nm in ("q_proj", "k_proj", "v_proj", "out_proj"):
            clip[lp + f"self_attn.{nm}.weight"] = big(C, C, C ** -0.5)
            clip[lp + f"self_attn.{nm}.bias"] = rn(C, std=0.02)
        clip[lp + "mlp.fc1.weight"] = big(CF, C, C ** -0.5); clip[lp + "mlp.fc1.bias"] = rn(CF, std=0.02)
        clip[lp + "mlp.fc2.weight"] = big(C, CF, CF ** -0.5); clip[lp + "mlp.fc2.bias"] = rn(C, std=0.02)
        for nm in ("layer_norm1", "layer_norm2"):
            clip[lp + nm + ".weight"] = 1 + rn(C, std=0.05); clip[lp + nm + ".bias"] = rn(C, std=0.02)
    llm = {"model.embed_tokens.weight": big(V, D, 1.0), "model.norm.weight": 1 + rn(D, std=0.05),
           "lm_head.weight": big(V, D, D ** -0.5),
           "model.mm_projector.weight": big(D, 1024, 1024 ** -0.5), "model.mm_projector.bias": rn(D, std=0.02)}
    for l in range(L):
        lp = f"model.layers.{l}."
        for nm in ("q_proj", "k_proj", "v_proj", "o_proj"):
            llm[lp + f"self_attn.{nm}.weight"] = big(D, D, D ** -0.5)
        llm[lp + "mlp.gate_proj.weight"] = big(F, D, D ** -0.5)
        llm[lp + "mlp.up_proj.weight"] = big(F, D, D ** -0.5)
        llm[lp + "mlp.down_proj.weight"] = big(D, F, F ** -0.5)
        llm[lp + "input_layernorm.weight"] = 1 + rn(D, std=0.05)
        llm[lp + "post_attention_layernorm.weight"] = 1 + rn(D, std=0.05)
    return clip, llm


def synthetic_prompt_ids(seed=1, n_pre=63, n_vid=356, n_post=26):
    """SURVEY.md section 8d, config 2: [1] + 63 ids ~ U[3,32000) + <vid_start> + <vid_patch> x 356 + <vid_end>
    + 26 ids ~ U[3,32000)  ->  S_p = 448 (ids 32000 / 32001 / 32002 are patch / start / end)."""
    g = torch.Generator().manual_seed(seed)
    pre = torch.randint(3, 32000, (n_pre,), generator=g)
    post = torch.randint(3, 32000, (n_post,), generator=g)
    row = torch.cat([torch.tensor([1]), pre, torch.tensor([32001]), torch.full((n_vid,), 32000), torch.tensor([32002]), post])
    return row[None].to(torch.int64)


def synthetic_frames(clip, t, size=224):
    return np.random.default_rng(1000 + clip).integers(0, 256, (t, size, size, 3), dtype=np.uint8)


def build_model(model, B, dev, clip_only=False):
    """The reference-facing objects (video_chatgpt.model mirror) over ONE libvcl handle, as
    initialize_model builds them (video_chatgpt/eval/model_utils.py:82-150), fed with random-init
    weights. Returns (model, tower, engine, (clip_sd, llm_sd))."""
    from video_chatgpt.model import VideoChatGPTConfig, VideoChatGPTLlamaForCausalLM
    m = MODELS[model]
    clip_sd, llm_sd = device_weights(model, dev)
    if clip_only:        # tower-only handle: a zero-layer language model keeps it small
        cfg = VideoChatGPTConfig(hidden_size=512, intermediate_size=1024, num_hidden_layers=0, num_attention_heads=4,
                                 vocab_size=8, use_mm_proj=True, mm_hidden_size=1024)
        llm_sd = None
    else:
        cfg = VideoChatGPTConfig(hidden_size=m["hidden"], intermediate_size=m["inter"], num_hidden_layers=m["layers"],
                                 num_attention_heads=m["heads"], vocab_size=32003, use_mm_proj=True, mm_hidden_size=1024,
                                 rms_norm_eps=1e-5, rope_theta=10000.0)
    mdl = VideoChatGPTLlamaForCausalLM(cfg, clip_config=dict(num_hidden_layers=24), max_batch=B,
                                       max_seq=S_PROMPT + N_NEW)
    vc = mdl.get_model().vision_config
    vc.vid_patch_token, vc.vid_start_token, vc.vid_end_token, vc.use_vid_start_end = 32000, 32001, 32002, True
    if llm_sd is not None:
        mdl.load_state_dict(llm_sd)
    tower = mdl.get_vision_tower()
    tower.load_state_dict(clip_sd)
    eng = mdl._ensure_engine(need_clip=True, need_llm=llm_sd is not None)
    return mdl, tower, eng, (clip_sd, llm_sd)


# ---------------------------------------------------------------------------------------------
# library baseline: the oracle in bf16 on this GPU through stock PyTorch kernels
# ---------------------------------------------------------------------------------------------
def library_sample(model, dev, clip_sd, llm_sd):
    """One clip of the headline workload (100 frames -> ViT -> pool -> 7B/13B prefill -> 32 greedy
    tokens) through oracle/vcl_oracle.py = the reference's op sequence on torch's own CUDA kernels
    (cuBLAS GEMMs; attention eager as the reference's HF code runs it, and SDPA as transformers 5.x
    would pick). The reference serves one clip at a time (inference.py:47-125), so this is batch 1."""
    from oracle import vcl_oracle as O
    m = MODELS[model]
    ccfg = O.ClipCfg()
    lcfg = O.LlmCfg(hidden=m["hidden"], inter=m["inter"], heads=m["heads"], layers=m["layers"])
    frames = torch.as_tensor(synthetic_frames(0, T_FRAMES)).to(dev)
    ids = synthetic_prompt_ids(seed=1).to(dev)
    mean = torch.tensor(O.CLIP_MEAN, device=dev)
    std = torch.tensor(O.CLIP_STD, device=dev)
    out = {"unit": "videos/s", "clips": 1, "dtype": "bf16",
           "what": "oracle/vcl_oracle.py (the reference's op sequence) on torch CUDA kernels, same GPU, 1 warm-up + 1 timed clip"}

    def one(attn):
        px = ((frames.float() * (1.0 / 255.0) - mean) / std).permute(0, 3, 1, 2).contiguous().bfloat16()
        hid = O.clip_hidden_states(clip_sd, ccfg, px, 23, attn=attn)[-1]
        feats = O.st_pool_torch(hid[:, 1:])
        toks, _ = O.greedy_generate(llm_sd, lcfg, ids, feats[None].bfloat16(), N_NEW, attn=attn)
        return toks

    with torch.no_grad():
        for attn in ("eager", "sdpa"):
            one(attn)
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            toks = one(attn)
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            out[attn] = {"value": 1.0 / dt, "ms_per_clip": dt * 1e3}
            out[attn + "_tokens"] = toks[0].tolist()
    return out


# ---------------------------------------------------------------------------------------------
# measured DRAM traffic of the decode loop, from the committed ncu capture
# ---------------------------------------------------------------------------------------------
def decode_traffic_from_ncu(model, B):
    """Measured DRAM bytes of the decode loop: profiles/r02_decode_step_traffic.json (tools/decode_traffic.py:
    dram__bytes_read + dram__bytes_write of every kernel of one decode step in an `ncu --set full` capture,
    per-layer part scaled to the model depth) x the steps of the loop. None when there is no capture for
    this configuration (7B, 1 clip)."""
    path = os.path.join(ROOT, "profiles", "r02_decode_step_traffic.json")
    if model != "7b" or B != 1 or not os.path.exists(path):
        return None, None
    try:
        d = json.load(open(path))
        return d["step_dram_bytes"] * (N_NEW - 1), os.path.relpath(path, ROOT) + " <- " + d["source"]
    except Exception:
        return None, None


# ---------------------------------------------------------------------------------------------
# product arm
# ---------------------------------------------------------------------------------------------
def init_dist(world, dev):
    if world <= 1:
        return None
    import torch.distributed as dist
    # keep stdout to the one JSON line: whatever NCCL logs (its version banner included) goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    dist.init_process_group("nccl", device_id=dev)
    return dist


def make_timer(dev, dist, step):
    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(k, n_events, *args):
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(n_events)] for _ in range(k)] if n_events else None
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(k):
            step(*args, evs[i] if evs else None)
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        if dist is not None:
            t = torch.tensor([ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = t.item()
        return ms, evs
    return timed


def run_vcl(args, rank, world, local_rank):
    import vcl_native as vn                 # the product arm never touches oracle/ inside the timed path
    from video_chatgpt.inference import get_spatio_temporal_features_torch
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    dist = init_dist(world, dev)
    m = MODELS[args.model]
    B = args.clips
    model, tower, eng, (clip_sd, llm_sd) = build_model(args.model, B, dev)
    want_library = rank == 0 and world == 1 and not args.no_library
    if not want_library:
        del clip_sd, llm_sd
        clip_sd = llm_sd = None
    torch.cuda.empty_cache()

    ids_h = synthetic_prompt_ids(seed=1).repeat(B, 1).pin_memory()
    vs_h = torch.full((B,), 64, dtype=torch.int32)
    frames_h = torch.stack([torch.as_tensor(synthetic_frames(rank * B + b, T_FRAMES)) for b in range(B)]).pin_memory()
    toks_h = torch.empty(B, N_NEW, dtype=torch.int32).pin_memory()
    frames_d, ids_d, vs_d = frames_h.to(dev), ids_h.to(dev), vs_h.to(dev)
    feats = torch.empty(B, 356, 1024, dtype=torch.bfloat16, device=dev)
    first = torch.empty(B, dtype=torch.int32, device=dev)
    toks = torch.empty(B, N_NEW, dtype=torch.int32, device=dev)
    gathered = torch.empty(world * B, N_NEW, dtype=torch.int32, device=dev) if world > 1 else None
    stream = torch.cuda.Stream(device=dev)
    h2d = frames_h.numel() + ids_h.numel() * 8
    d2h = toks_h.numel() * 4

    def step(host_io, ev=None):
        if host_io:
            # the reference caller's sequence (video_chatgpt/inference.py:86-112) on the mirror API,
            # from pinned host buffers; the image processor's normalisation runs on the device
            # (raw uint8 frames go in), everything else is the reference's own call surface
            fl = []
            for b in range(B):
                outs = tower(frames_h[b].to(dev, non_blocking=True), output_hidden_states=True)
                fl.append(get_spatio_temporal_features_torch(outs.hidden_states[-2][:, 1:]))
            out = model.generate(ids_h.to(dev, non_blocking=True), video_spatio_temporal_features=torch.stack(fl),
                                 do_sample=False, max_new_tokens=N_NEW, eos_token_id=None)
            new = out[:, S_PROMPT:].to(torch.int32).contiguous()
            if gathered is not None:
                dist.all_gather_into_tensor(gathered, new)
            toks_h.copy_(gathered[:B] if gathered is not None else new, non_blocking=True)
            return
        if ev: ev[0].record()
        for b in range(B):
            eng.clip_features(frames_d[b], out=feats[b])
        if ev: ev[1].record()
        eng.prefill(ids_d, feats, vs_d, tok_out=first)
        if ev: ev[2].record()
        eng.decode_loop(first, S_PROMPT, N_NEW, out=toks)
        if ev: ev[3].record()
        if gathered is not None:
            dist.all_gather_into_tensor(gathered, toks)

    timed = make_timer(dev, dist, step)
    clocks = Clocks(local_rank)
    warm = max(args.warmup, 3)
    with torch.cuda.stream(stream):
        for _ in range(warm):
            step(True)
        for _ in range(2):
            step(False)
        l0 = vn.launch_count()
        clocks.start()
        ms_dev, evs = timed(args.steps, 4, False)
        launches = vn.launch_count() - l0
        outputs = {"tokens": (gathered if gathered is not None else toks).clone(),
                   "video_features": feats.clone()} if args.dump_outputs and rank == 0 else None
        ms_e2e, _ = timed(args.steps, 0, True)
        clk = clocks.stop()
        stream.synchronize()
        api_tokens = toks_h.clone()
        agree = bool(torch.equal(api_tokens, toks.cpu()))
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    stage = np.array([[ev[i].elapsed_time(ev[i + 1]) for i in range(3)] for ev in evs]).mean(0)  # ms: clip, prefill, decode

    w = work(args.model)
    hbm, tf, src = peaks()
    dec_bytes = (N_NEW - 1) * w["weights_step"] + B * w["kv_per_tok"] * sum(S_PROMPT + i for i in range(1, N_NEW))
    dec_gbs = dec_bytes / (stage[2] * 1e-3) / 1e9
    traffic, traffic_src = decode_traffic_from_ncu(args.model, B)
    total_clips = world * B * args.steps
    out = {
        "metric": metric_name(args.config, args.model),
        "value": total_clips / (ms_dev * 1e-3), "unit": "videos/s", "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args.config, args.model, B, world),
        "e2e": {"value": total_clips / (ms_e2e * 1e-3), "unit": "videos/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e / args.steps,
                "api": "vision_tower(frames).hidden_states[-2][:, 1:] -> get_spatio_temporal_features_torch -> "
                       "model.generate (the video_chatgpt mirror), pinned host buffers",
                "tokens_equal_device_resident_run": agree},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": dec_gbs, "peak": hbm, "unit": "GB/s", "frac": dec_gbs / hbm,
                     "traffic": traffic,
                     "traffic_note": ("dram__bytes_read+write summed over the kernels of one decode step in the committed "
                                      f"ncu --set full capture ({traffic_src}) x {N_NEW - 1} steps; algorithmic bytes "
                                      f"{dec_bytes / 1e9:.1f} GB") if traffic else "no committed ncu capture for this configuration",
                     "peak_source": src,
                     "kernel": f"decode loop: {N_NEW - 1} steps x (4 weight-streaming launches + attention per layer x "
                               f"{m['layers']} layers + head), one CUDA graph; bytes = weights streamed + KV read"},
        "stages": {"clip_ms": stage[0], "prefill_ms": stage[1], "decode_ms": stage[2],
                   "clip_tflops": B * w["vit_flops"] / (stage[0] * 1e-3) / 1e12,
                   "prefill_tflops": B * w["prefill_flops"] / (stage[1] * 1e-3) / 1e12,
                   "tensor_peak_tflops": tf, "clip_frac": B * w["vit_flops"] / (stage[0] * 1e-3) / 1e12 / tf,
                   "prefill_frac": B * w["prefill_flops"] / (stage[1] * 1e-3) / 1e12 / tf},
        "clocks": clk,
    }
    if rank == 0:
        out["tokens_rank0_clip0"] = toks[0].tolist()
        if want_library:
            lib = library_sample(args.model, dev, clip_sd, llm_sd)
            # the product's greedy ids next to the library path's on the same weights and inputs
            lib["vcl_tokens_equal_eager"] = lib["eager_tokens"] == out["tokens_rank0_clip0"]
            lib["vcl_tokens_equal_sdpa"] = lib["sdpa_tokens"] == out["tokens_rank0_clip0"]
            n_agree = sum(int(a == b) for a, b in zip(lib["eager_tokens"], out["tokens_rank0_clip0"]))
            lib["vcl_vs_eager_first_tokens_identical"] = next((i for i, (a, b) in enumerate(
                zip(lib["eager_tokens"], out["tokens_rank0_clip0"])) if a != b), N_NEW)
            lib["vcl_vs_eager_agreement"] = n_agree / N_NEW
            per_clip_ms = ms_e2e / args.steps / B
            lib["vcl_speedup_vs_eager"] = lib["eager"]["ms_per_clip"] / per_clip_ms
            lib["vcl_speedup_vs_sdpa"] = lib["sdpa"]["ms_per_clip"] / per_clip_ms
            out["library_baseline"] = lib
            del clip_sd, llm_sd
        if world == 1 and not args.no_cpu:
            out["cpu_baseline"] = cpu_sample(args.model)
        emit(out)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------
# config 5: CLIP-only extraction sweep (the GPU replacement of the reference's offline extractor loop,
# scripts/save_spatio_temporal_clip_features.py:95-139)
# ---------------------------------------------------------------------------------------------
def run_clip_sweep(args, rank, world, local_rank):
    import vcl_native as vn
    from video_chatgpt.inference import get_spatio_temporal_features_torch
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    dist = init_dist(world, dev)
    _, tower, eng, _ = build_model("7b", 1, dev, clip_only=True)
    torch.cuda.empty_cache()
    Ts = [int(t) for t in args.frames.split(",")]
    frames_h = {t: torch.as_tensor(synthetic_frames(rank, t)).pin_memory() for t in Ts}
    frames_d = {t: frames_h[t].to(dev) for t in Ts}
    outs = {t: torch.empty(356, 1024, dtype=torch.float16, device=dev) for t in Ts}
    sums = torch.zeros(len(Ts), dtype=torch.float32, device=dev)
    sums_h = torch.empty(world * len(Ts), dtype=torch.float32).pin_memory()
    gathered = torch.empty(world * len(Ts), dtype=torch.float32, device=dev)
    stream = torch.cuda.Stream(device=dev)

    def step(host_io, ev=None):
        for i, t in enumerate(Ts):
            if ev: ev[i].record()
            if host_io:
                hs = tower(frames_h[t].to(dev, non_blocking=True), output_hidden_states=True).hidden_states[-2][:, 1:]
                feats = get_spatio_temporal_features_torch(hs)
            else:
                feats = eng.clip_features(frames_d[t], out=outs[t])
            sums[i] = feats.float().sum()             # per-clip checksum (what the gather carries)
        if ev: ev[len(Ts)].record()
        if dist is not None:
            dist.all_gather_into_tensor(gathered, sums)
        if host_io:
            sums_h.copy_(gathered if dist is not None else sums, non_blocking=True)

    timed = make_timer(dev, dist, step)
    clocks = Clocks(local_rank)
    warm = max(args.warmup, 3)
    with torch.cuda.stream(stream):
        for _ in range(warm):
            step(True)
        step(False)
        l0 = vn.launch_count()
        clocks.start()
        ms_dev, evs = timed(args.steps, len(Ts) + 1, False)
        launches = vn.launch_count() - l0
        outputs = {f"video_features_T{t}": outs[t].clone() for t in Ts} if args.dump_outputs and rank == 0 else None
        ms_e2e, _ = timed(args.steps, 0, True)
        clk = clocks.stop()
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    per_t = np.array([[ev[i].elapsed_time(ev[i + 1]) for i in range(len(Ts))] for ev in evs]).mean(0)   # ms per clip at each T
    hbm, tf, src = peaks()
    sweep = {}
    for i, t in enumerate(Ts):
        tfl = VIT_FLOPS_PER_FRAME * t / (per_t[i] * 1e-3) / 1e12
        sweep[str(t)] = {"ms_per_clip": per_t[i], "clips_per_s_per_gpu": 1e3 / per_t[i], "tflops": tfl, "frac_of_tensor_peak": tfl / tf,
                         "job_seconds_1000_clips": SWEEP_CLIPS * per_t[i] * 1e-3 / world}
    total_clips = world * len(Ts) * args.steps
    flops_step = VIT_FLOPS_PER_FRAME * sum(Ts)
    ach = flops_step / (per_t.sum() * 1e-3) / 1e12
    out = {
        "metric": metric_name(5, "7b"), "value": total_clips / (ms_dev * 1e-3), "unit": "videos/s", "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(5, "7b", 1, world),
        "e2e": {"value": total_clips / (ms_e2e * 1e-3), "unit": "videos/s",
                "h2d_bytes_per_step": int(sum(frames_h[t].numel() for t in Ts)), "d2h_bytes_per_step": int(sums_h.numel() * 4),
                "ms_per_step": ms_e2e / args.steps,
                "api": "vision_tower(frames).hidden_states[-2][:, 1:] -> get_spatio_temporal_features_torch, pinned host frames"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "achieved": ach, "peak": tf, "unit": "TFLOP/s", "frac": ach / tf, "traffic": None,
                     "peak_source": src, "kernel": "the ViT's tcgen05 GEMMs + attention over one clip (algorithmic flops of SURVEY.md 8d / clip time)"},
        "sweep": sweep,
        "job": {"clips_per_T": SWEEP_CLIPS, "seconds_for_the_whole_sweep": sum(v["job_seconds_1000_clips"] for v in sweep.values())},
        "clocks": clk,
    }
    if rank == 0:
        emit(out)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------
# the other arms
# ---------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path on the box's host cores (the oracle port:
    the reference is pure Python over HF / PyTorch and cannot be installed offline). ONE bounded sample
    (about 1-2 minutes) independent of --steps / --warmup; rank 0 only."""
    if rank != 0:
        return
    s = cpu_sample(args.model)
    v = s["value"]
    emit({
        "impl": "reference", "metric": metric_name(args.config, args.model), "value": v, "unit": "videos/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": s["dtype"], "data": "synthetic",
        "config": workload_config(args.config, args.model, args.clips, world),
        "cpu_baseline": s,
        "e2e": {"value": v, "unit": "videos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "one bounded CPU sample extrapolated to one clip of the configured workload (see cpu_baseline.sample); "
                "the CPU arm serves one clip at a time, as the reference does",
    })


def run_library(args, rank, world, local_rank):
    if rank != 0:
        return
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    clip_sd, llm_sd = device_weights(args.model, dev)
    lib = library_sample(args.model, dev, clip_sd, llm_sd)
    emit({"impl": "library", "metric": metric_name(args.config, args.model), "value": lib["eager"]["value"],
          "unit": "videos/s", "n_gpus": 1, "higher_is_better": True, "dtype": "bf16", "data": "synthetic",
          "config": workload_config(args.config, args.model, 1, 1), "library_baseline": lib})


_REAL_STDOUT = None


def emit(obj):
    """The ONE JSON line of the contract, written to the process's real stdout."""
    line = json.dumps(obj) + "\n"
    if _REAL_STDOUT is None:
        sys.stdout.write(line); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line.encode())


def main():
    # stdout carries the JSON line and nothing else: whatever libraries print meanwhile (NCCL's version banner
    # on some boxes, warnings) is sent to stderr by pointing fd 1 at fd 2 for the duration of the run
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vcl", choices=["vcl", "reference", "library"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="SURVEY.md 8d configuration (2 = headline)")
    ap.add_argument("--clips", type=int, default=None, help="clips per GPU per step (default: the configuration's)")
    ap.add_argument("--model", default=None, choices=list(MODELS))
    ap.add_argument("--frames", default="32,64,100", help="config 5: frames per clip, comma separated")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-library", action="store_true", help="skip the library_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "vcl":
        ap.error("--dump-outputs needs --impl vcl")
    if args.model is None:
        args.model = CONFIGS[args.config]["model"]
    if args.clips is None:
        args.clips = CONFIGS[args.config]["clips"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.impl == "library":
        run_library(args, rank, world, local_rank)
    elif args.config == 5:
        run_clip_sweep(args, rank, world, local_rank)
    else:
        run_vcl(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
