"""Decode cost of sampling and stopping criteria, per generated token, on the headline shapes.

    python tools/sampling_bench.py [--model 7b] [--batches 1,16] [--n-new 64] [--repeats 3] [--out FILE]

Config-2 shapes (Vicuna-7B with random-init weights, S_p = 448 prompt tokens, 356 video rows), EOS disabled
so that every run decodes exactly n_new tokens (default 64: every position stays below 512 keys, the range the
GPU tests cover), on a side stream. For each batch size it times whole
generate() calls of four kinds and reports (call time - prefill time) / (n_new - 1) as ms per token:

    greedy            do_sample=False: one CUDA-graph decode loop
    device_sampled    do_sample=True, temperature 0.2, top-k 50: sampled graph loops of 32 tokens
    host_sampling     the same call with VCL_HOST_SAMPLING=1: one C-ABI step + torch sampling per token
    infer_settings    video_chatgpt_infer's settings (do_sample, temperature 0.2, top-k 50) with its stop-string
                      criterion (KeywordsStoppingCriteria), over a stand-in tokenizer whose batch_decode spells
                      ids as words, so the criterion never fires and the run keeps its length

and the sampler kernel on its own ([B, 32003] fp32 logits, CUDA events over 200 launches). Prints one JSON
object (also written to --out).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "video-llava_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import bench  # noqa: E402  (weights and prompt of the benchmark's workload)


class _WordTokenizer:
    """Stand-in for the LLaMA tokenizer: "</s>" is not a single id, batch_decode spells ids as words."""

    def __call__(self, text):
        return type("E", (), {"input_ids": [1, 2]})()

    def batch_decode(self, ids, skip_special_tokens=True):
        return [" ".join(f"w{int(t)}" for t in row) for row in ids.tolist()]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def build(model, B, max_seq, dev):
    from video_chatgpt.model import VideoChatGPTConfig, VideoChatGPTLlamaForCausalLM
    m = bench.MODELS[model]
    _, llm_sd = bench.device_weights(model, dev)
    cfg = VideoChatGPTConfig(hidden_size=m["hidden"], intermediate_size=m["inter"], num_hidden_layers=m["layers"],
                             num_attention_heads=m["heads"], vocab_size=32003, use_mm_proj=True, mm_hidden_size=1024)
    mdl = VideoChatGPTLlamaForCausalLM(cfg, clip_config=dict(num_hidden_layers=24), max_batch=B, max_seq=max_seq)
    vc = mdl.get_model().vision_config
    vc.vid_patch_token, vc.vid_start_token, vc.vid_end_token, vc.use_vid_start_end = 32000, 32001, 32002, True
    mdl.load_state_dict(llm_sd)
    eng = mdl._ensure_engine(need_llm=True)
    del llm_sd
    torch.cuda.empty_cache()
    return mdl, eng


def timed(fn, repeats, st):
    ts = []
    for _ in range(repeats):
        st.synchronize()
        t0 = time.perf_counter()
        fn()
        st.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def kernel_time(logits, T, k, st, n=200):
    import vcl_native as vn
    with torch.cuda.stream(st):
        for i in range(10):
            vn.op_sample(logits, T, k, 1, 448 + i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for i in range(n):
            vn.op_sample(logits, T, k, 1, 448 + i)
        e1.record(st)
    st.synchronize()
    return e0.elapsed_time(e1) / n * 1e3          # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="7b", choices=list(bench.MODELS))
    ap.add_argument("--batches", default="1,16")
    ap.add_argument("--n-new", type=int, default=64)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sampling_bench.py needs a GPU")
    from video_chatgpt.model.utils import KeywordsStoppingCriteria
    dev = torch.device("cuda:0")
    n = args.n_new
    res = {"gpu": gpu_info(), "model": args.model, "S_prompt": bench.S_PROMPT, "n_new": n, "eos": None,
           "repeats": args.repeats, "statistic": "median", "batches": {}}
    st = torch.cuda.Stream()
    for B in [int(b) for b in args.batches.split(",")]:
        mdl, eng = build(args.model, B, bench.S_PROMPT + n, dev)
        ids = bench.synthetic_prompt_ids().expand(B, -1).contiguous().to(dev)
        feats = (torch.randn(B, 356, 1024, generator=torch.Generator().manual_seed(B)) * 0.5).half().to(dev)
        vs = mdl._spans_dev(ids, feats, eng.NV)
        kinds = {
            "greedy": (dict(do_sample=False), False, False),
            "device_sampled": (dict(do_sample=True, temperature=0.2, top_k=50), False, False),
            "host_sampling": (dict(do_sample=True, temperature=0.2, top_k=50), True, False),
            "infer_settings": (dict(do_sample=True, temperature=0.2, top_k=50), False, True),
        }
        row = {}
        with torch.cuda.stream(st):
            t_pre = timed(lambda: eng.prefill(ids, feats, vs, want_logits=True, want_token=False), args.repeats + 1, st)
            row["prefill_ms"] = round(t_pre * 1e3, 3)
            for name, (kw, host, crit) in kinds.items():
                def run():
                    c = [KeywordsStoppingCriteria(["</s>"], _WordTokenizer(), ids)] if crit else None
                    out = mdl.generate(ids, video_spatio_temporal_features=feats, max_new_tokens=n, eos_token_id=None,
                                       stopping_criteria=c, **kw)
                    assert out.shape == (B, bench.S_PROMPT + n), out.shape
                print(f"[sampling_bench] B={B} {name}", file=sys.stderr, flush=True)
                if host:
                    os.environ["VCL_HOST_SAMPLING"] = "1"
                try:
                    run()                                  # warm-up: graphs captured, kernels loaded
                    t = timed(run, args.repeats, st)
                finally:
                    os.environ.pop("VCL_HOST_SAMPLING", None)
                row[name] = {"call_ms": round(t * 1e3, 2), "ms_per_token": round((t - t_pre) * 1e3 / (n - 1), 4)}
        g = row["greedy"]["ms_per_token"]
        for name in kinds:
            row[name]["vs_greedy"] = round(row[name]["ms_per_token"] / g, 4)
        logits = torch.randn(B, 32003, generator=torch.Generator().manual_seed(0)).bfloat16().float().to(dev)
        row["sample_kernel_us"] = {"T0.2_k50": round(kernel_time(logits, 0.2, 50, st), 2),
                                   "T1_k0": round(kernel_time(logits, 1.0, 0, st), 2),
                                   "T0_argmax": round(kernel_time(logits, 0.0, 50, st), 2)}
        res["batches"][str(B)] = row
        print(json.dumps({"B": B, **row}), file=sys.stderr)
        del mdl, eng
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
