"""The reference-facing Python surface (video_chatgpt.* mirror) on the GPU: same calls the
reference's callers make (inference.py:93-120, scripts/save_spatio_temporal_clip_features.py),
checked against the golden fixtures and the oracle."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import vcl_oracle as O  # noqa: E402

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _model(llm_cfg, clip_layers_total=3, max_batch=2):
    from video_chatgpt.model import VideoChatGPTConfig, VideoChatGPTLlamaForCausalLM
    cfg = VideoChatGPTConfig(hidden_size=llm_cfg.hidden, intermediate_size=llm_cfg.inter,
                             num_hidden_layers=llm_cfg.layers, num_attention_heads=llm_cfg.heads,
                             vocab_size=llm_cfg.vocab, use_mm_proj=True, mm_hidden_size=1024)
    clip = dict(hidden_size=1024, intermediate_size=1024, num_hidden_layers=clip_layers_total, num_attention_heads=16)
    m = VideoChatGPTLlamaForCausalLM(cfg, clip_config=clip, max_batch=max_batch, max_seq=480)
    vc = m.get_model().vision_config
    vc.vid_patch_token, vc.vid_start_token, vc.vid_end_token, vc.use_vid_start_end = 32000, 32001, 32002, True
    return m


def test_pool_functions_vs_reference_fixtures():
    from video_chatgpt.inference import get_spatio_temporal_features_torch
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "vcl_save_feats", os.path.join(os.path.dirname(G), "..", "video-llava_b200", "scripts",
                                       "save_spatio_temporal_clip_features.py"))
    mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
    from _util import load_pool_golden
    g = load_pool_golden(os.path.join(G, "pool.npz"))
    gen = torch.Generator().manual_seed(5)
    f8 = torch.randn(8, 256, 1024, generator=gen).half()
    f100 = torch.randn(100, 256, 1024, generator=gen).half()
    o8 = get_spatio_temporal_features_torch(f8.cuda())
    assert o8.dtype == torch.float16 and o8.shape == (356, 1024) and o8.is_cuda
    assert (o8[8:100] == 0).all()
    for ours, ref in [(o8.cpu().numpy(), g["t8_torch"]),
                      (mod.get_spatio_temporal_features(f8.numpy()), g["t8_numpy"]),
                      (get_spatio_temporal_features_torch(f100.cuda()).cpu().numpy()[::7], g["t100_torch_rows"]),
                      (get_spatio_temporal_features_torch(f100.bfloat16().cuda()).cpu().numpy()[::7], g["t100_bf16_rows"])]:
        assert ours.dtype == np.float16 and ours.shape == ref.shape
        d = np.abs(ours.astype(np.float32) - ref.astype(np.float32))
        ulp = np.maximum(np.abs(ref.astype(np.float32)), 2.0 ** -14) * 2.0 ** -10
        # fp32 summation order differs from torch's / numpy's trees: <= 1 ulp of the output, mostly exact
        assert (d <= ulp).all(), d.max()
        assert (ours == ref).mean() > 0.97


@torch.no_grad()
def test_tower_pool_generate_like_the_reference_caller():
    from video_chatgpt.inference import get_spatio_temporal_features_torch
    from video_chatgpt.model.utils import KeywordsStoppingCriteria
    lcfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2)
    ccfg = O.ClipCfg(hidden=1024, inter=1024, heads=16, layers=3)
    m = _model(lcfg, 3, max_batch=1)
    lsd, csd = O.random_llm_state(lcfg, seed=21), O.random_clip_state(ccfg, seed=11)
    m.load_state_dict(lsd)
    tower = m.get_vision_tower()
    tower.load_state_dict(csd)
    px = O.preprocess_frames(O.make_frames(7, 3))
    outs = tower(px.half().cuda(), output_hidden_states=True)
    assert len(outs.hidden_states) == 4
    feats_in = outs.hidden_states[-2][:, 1:]
    assert feats_in.shape == (3, 256, 1024)
    with pytest.raises(Exception, match="needs encoder layer 3"):
        outs.hidden_states[-1]
    feats = get_spatio_temporal_features_torch(feats_in)
    assert feats.shape == (356, 1024) and feats.dtype == torch.float16
    ids = O.make_prompt_ids(lcfg, 356, seed=1).cuda()
    out = m.generate(ids, video_spatio_temporal_features=feats.unsqueeze(0), do_sample=False, max_new_tokens=6)
    assert out.shape == (1, 448 + 6) and out.dtype == torch.int64
    assert torch.equal(out[:, :448], ids)                           # prompt included, like HF generate
    bf = lambda sd: {k: v.cuda().bfloat16() for k, v in sd.items()}
    ref_toks, ref_logits = O.greedy_generate(bf(lsd), lcfg, ids, feats[None].bfloat16(), 6)
    lg = m(input_ids=ids, video_spatio_temporal_features=feats.unsqueeze(0)).logits
    assert lg.shape == (1, 1, lcfg.vocab)
    rel = ((lg[:, 0].float() - ref_logits[0]).norm() / ref_logits[0].norm()).item()
    assert rel < 3e-2, rel
    assert out[0, 448].item() == ref_toks[0, 0].item()
    # cached single-token step through forward(), as HF's generation loop drives it
    step = m(input_ids=out[:, 448:449], past_key_values=448, video_spatio_temporal_features=feats.unsqueeze(0)).logits
    assert step[:, 0].argmax(-1).item() == out[0, 449].item()

    class Tok:   # stop on token id == the third generated token
        def __init__(self, stop): self.stop = stop
        def __call__(self, text): return type("E", (), {"input_ids": [self.stop]})()
        def batch_decode(self, ids, skip_special_tokens=True): return [""]
    crit = KeywordsStoppingCriteria(["x"], Tok(int(out[0, 450])), ids)
    out2 = m.generate(ids, video_spatio_temporal_features=feats.unsqueeze(0), do_sample=False, max_new_tokens=6,
                      stopping_criteria=[crit])
    assert out2.shape[1] == 448 + 3 and torch.equal(out2, out[:, :451])
    out3 = m.generate(ids, video_spatio_temporal_features=feats.unsqueeze(0), do_sample=True, temperature=0.2,
                      max_new_tokens=4)
    assert out3.shape == (1, 452)
    bad = ids.clone(); bad[0, 64 + 357] = 5
    with pytest.raises(ValueError, match="video start tokens and video end tokens"):
        m.generate(bad, video_spatio_temporal_features=feats.unsqueeze(0), max_new_tokens=2)


@torch.no_grad()
def test_generate_continue_second_turn():
    """Second turn about the same video through the KV cache (generate_continue): the tokens it
    produces must be the ones a from-scratch pass over the concatenated context decides on."""
    lcfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2)
    m = _model(lcfg, 3, max_batch=1)
    m.load_state_dict(O.random_llm_state(lcfg, seed=23))
    feats = (torch.randn(356, 1024, generator=torch.Generator().manual_seed(3)) * 0.5).half().cuda()
    ids = O.make_prompt_ids(lcfg, 356, seed=2).cuda()
    turn1 = m.generate(ids, video_spatio_temporal_features=feats.unsqueeze(0), do_sample=False, max_new_tokens=5)
    q2 = torch.randint(3, 32000, (1, 11), generator=torch.Generator().manual_seed(8)).cuda()
    turn2 = m.generate_continue(q2, do_sample=False, max_new_tokens=5)
    assert turn2.shape == (1, 448 + 5 + 11 + 5)
    assert torch.equal(turn2[:, :453], turn1) and torch.equal(turn2[:, 453:464], q2)
    # The same context from scratch, teacher-forced with the continued turn's tokens (a free-running comparison
    # says nothing after the first near-tie): the two paths share the arithmetic up to the GEMM / GEMV tiling
    # that produced the cached rows, so every continued token must be the from-scratch arg-max wherever that
    # arg-max is decided by >= 3 bf16 ulps, and one of the tied candidates otherwise.
    n_strict = 0
    for i in range(5):
        ctx = turn2[:, :464 + i]
        lg = m(input_ids=ctx, video_spatio_temporal_features=feats.unsqueeze(0)).logits[0, -1].float()
        top = torch.topk(lg, 2)
        ulp = top.values[0].abs().clamp_min(2 ** -6) * 2 ** -7
        margin = ((top.values[0] - top.values[1]) / ulp).item()
        gap = ((top.values[0] - lg[turn2[0, 464 + i]]) / ulp).item()
        print(f"[dropin] second turn, token {i}: continued {turn2[0, 464 + i].item()} from-scratch arg-max "
              f"{top.indices[0].item()} (margin {margin:.1f} ulps, continued token {gap:.1f} ulps below the top)")
        if margin >= 3:
            n_strict += 1
            assert gap == 0, (i, margin, gap)
        else:
            assert gap < 3, (i, margin, gap)
    assert n_strict >= 1
    m2 = _model(lcfg, 3, max_batch=1)
    with pytest.raises(ValueError, match="no previous generate"):
        m2.generate_continue(q2)


@torch.no_grad()
def test_generate_stops_at_eos_per_row_like_hf():
    """ADVICE r1 (high): generate() honours EOS by default. Two clips whose greedy continuations hit the
    chosen EOS id at different steps: each row is padded after ITS EOS, the call returns when both are
    done, greedy chunks on the device and the stepwise (sampling-style) path agree."""
    lcfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2)
    m = _model(lcfg, 3, max_batch=2)
    m.load_state_dict(O.random_llm_state(lcfg, seed=21))
    feats = (torch.randn(2, 356, 1024, generator=torch.Generator().manual_seed(4)) * 0.5).half().cuda()
    ids = O.make_prompt_ids(lcfg, 356, seed=3, batch=2).cuda()
    free = m.generate(ids, video_spatio_temporal_features=feats, do_sample=False, max_new_tokens=24, eos_token_id=None)
    assert free.shape == (2, 448 + 24)
    new = free[:, 448:]
    eos = int(new[0, 5])                                   # row 0 finishes at step 5 (or earlier if repeated)
    first = [int((new[b] == eos).nonzero()[0]) if (new[b] == eos).any() else None for b in range(2)]
    out = m.generate(ids, video_spatio_temporal_features=feats, do_sample=False, max_new_tokens=24, eos_token_id=eos,
                     pad_token_id=0)
    got = out[:, 448:]
    if first[1] is None:                                   # row 1 never emits it: runs to the limit
        assert got.shape[1] == 24
    else:
        assert got.shape[1] == max(first) + 1
    for b in range(2):
        k = first[b] if first[b] is not None else got.shape[1] - 1
        assert torch.equal(got[b, : k + 1], new[b, : k + 1])           # identical up to and including the EOS
        assert (got[b, k + 1:] == 0).all()                              # padded afterwards
    # the per-token path (what sampling / stopping criteria use) gives the same sequences
    class Never:
        def __call__(self, *a, **k): return False
    out2 = m.generate(ids, video_spatio_temporal_features=feats, do_sample=False, max_new_tokens=24, eos_token_id=eos,
                      pad_token_id=0, stopping_criteria=[Never()])
    assert torch.equal(out2, out)
    # default = config.eos_token_id (2 for LLaMA): a model that never emits 2 decodes max_new_tokens
    assert m._eos_pad("config", None)[0] == 2


@torch.no_grad()
def test_forward_hidden_states_like_hf():
    """forward(output_hidden_states=True) (reference video_chatgpt.py:205-218 over HF LlamaModel): L+1
    tensors from one pass, the LAST one after the final RMSNorm, against the oracle."""
    lcfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2)
    m = _model(lcfg, 3, max_batch=2)
    lsd = O.random_llm_state(lcfg, seed=21)
    m.load_state_dict(lsd)
    feats = (torch.randn(2, 356, 1024, generator=torch.Generator().manual_seed(9)) * 0.5).half().cuda()
    ids = O.make_prompt_ids(lcfg, 356, seed=1, batch=2).cuda()
    out = m(input_ids=ids, video_spatio_temporal_features=feats, output_hidden_states=True)
    assert len(out.hidden_states) == 3 and out.logits.shape == (2, 1, lcfg.vocab)
    bf = {k: v.cuda().bfloat16() for k, v in lsd.items()}
    f32 = {k: v.cuda().float() for k, v in lsd.items()}
    _, ref_hs, _ = O.llm_forward(bf, lcfg, ids, feats.bfloat16())
    _, gold_hs, _ = O.llm_forward(f32, lcfg, ids, feats.float())
    from _util import bar
    for i in range(3):
        assert out.hidden_states[i].shape == (2, 448, 512)
        bar(out.hidden_states[i], ref_hs[i], gold_hs[i], f"forward().hidden_states[{i}]" + (" (post-norm)" if i == 2 else ""))


@torch.no_grad()
def test_initialize_model_and_video_chatgpt_infer_end_to_end(tmp_path):
    """The drop-in entry points themselves (reference eval/model_utils.py:82-150, inference.py:47-125) on a
    synthetic LOCAL checkpoint: tokenizer + config + safetensors + CLIP directory -> initialize_model ->
    video_chatgpt_infer (PIL frames, image processor, tower, pool, generate with stop string and EOS,
    decode), against the same steps done with the oracle."""
    from PIL import Image
    from _checkpoint import make_tiny_checkpoint
    from video_chatgpt.eval.model_utils import initialize_model
    from video_chatgpt.inference import video_chatgpt_infer
    from video_chatgpt.video_conversation import conv_templates
    ck = make_tiny_checkpoint(tmp_path)
    model, tower, tok, ip, vlen = initialize_model(ck["model_dir"], max_batch=1, max_seq=1024)
    assert vlen == 356 and len(tok) == 1003
    vc = model.get_model().vision_config
    assert (vc.vid_patch_token, vc.vid_start_token, vc.vid_end_token, vc.use_vid_start_end) == (1000, 1001, 1002, True)
    assert model.state_dict()["model.embed_tokens.weight"].shape[0] == 1003 and model.config.vocab_size == 1003
    frames = [Image.fromarray(f) for f in O.make_frames(21, 6)]
    question = "w10 w11 w12 w13"
    text = video_chatgpt_infer(frames, question, "pg-video-llava", model, tower, tok, ip, vlen, do_sample=False,
                               max_new_tokens=10)
    assert isinstance(text, str)

    # the same steps with the oracle on the same (resized) weights
    conv = conv_templates["pg-video-llava"].copy()
    conv.append_message(conv.roles[0], question + "\n" + "<vid_start>" + "<vid_patch>" * vlen + "<vid_end>")
    conv.append_message(conv.roles[1], None)
    ids = torch.as_tensor(tok([conv.get_prompt()]).input_ids).cuda()
    assert (ids == 1000).sum() == 356 and (ids == 1001).sum() == 1 and ids[0, 0] == 1
    px = ip.preprocess(frames, return_tensors="pt")["pixel_values"].cuda().bfloat16()
    csd = {k: v.cuda().bfloat16() for k, v in ck["clip_sd"].items()}
    hid = O.clip_hidden_states(csd, ck["clip_cfg"], px, 2)[-1]
    feats = O.st_pool_torch(hid[:, 1:])
    lsd = {k: v.cuda().bfloat16() for k, v in model.state_dict().items()}
    lcfg = O.LlmCfg(hidden=512, inter=1024, heads=4, layers=2, vocab=1003, vid_patch_token=1000, vid_start_token=1001,
                    vid_end_token=1002)
    o_toks, o_logits = O.greedy_generate(lsd, lcfg, ids, feats[None].bfloat16(), 10)
    row = o_toks[0].tolist()
    if 2 in row:
        row = row[: row.index(2) + 1]
    want = tok.batch_decode([row], skip_special_tokens=True)[0].strip()
    top = torch.topk(o_logits[:, 0], 2, dim=-1).values
    margins = (top[:, 0] - top[:, 1]) / (top[:, 0].abs().clamp_min(2 ** -6) * 2 ** -7)
    print(f"[dropin] video_chatgpt_infer -> {text!r}; oracle -> {want!r}; min oracle margin {margins.min().item():.1f} ulps")
    assert text.split()[:1] == want.split()[:1]
    if margins.min() >= 3:
        assert text == want


def test_offline_extractor_main_format_resume_and_flush(tmp_path, monkeypatch):
    """scripts/save_spatio_temporal_clip_features.py:main (reference :95-139) with a `decord` stub: one
    pickle of a [356,1024] float16 ndarray per video, videos that already have a pickle are skipped,
    pending features are written every FLUSH_EVERY processed videos and at the end; the features equal
    the reference's numpy pooling of the tower's hidden state, and the training-side reader loads them."""
    import importlib.util
    import pickle
    import sys
    import types
    from _checkpoint import make_tiny_checkpoint
    ck = make_tiny_checkpoint(tmp_path)
    vids, outd = tmp_path / "videos", tmp_path / "feats"
    vids.mkdir()
    clips = {f"clip{i}": O.make_frames(40 + i, 4 + i) for i in range(4)}         # 4..7 frames each
    for name, fr in clips.items():
        np.save(vids / f"{name}.npy", fr)
    (vids / "broken.npy").write_bytes(b"not a video")
    seen_at_open = {}

    class VideoReader:                       # decord.VideoReader over .npy "videos"
        def __init__(self, path, ctx=None):
            seen_at_open[os.path.basename(path)] = sorted(os.listdir(outd))
            self.arr = np.load(path)
        def __len__(self): return len(self.arr)
        def get_batch(self, idx): return types.SimpleNamespace(asnumpy=lambda: self.arr[list(idx)])
    monkeypatch.setitem(sys.modules, "decord", types.SimpleNamespace(VideoReader=VideoReader, cpu=lambda i: None))
    spec = importlib.util.spec_from_file_location(
        "vcl_save_feats_main", os.path.join(os.path.dirname(G), "..", "video-llava_b200", "scripts",
                                            "save_spatio_temporal_clip_features.py"))
    mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
    outd.mkdir()
    with open(outd / "clip1.pkl", "wb") as f:                                   # "already processed": must be skipped
        pickle.dump("sentinel", f)
    monkeypatch.setattr(mod, "FLUSH_EVERY", 2)
    monkeypatch.setattr(sys, "argv", ["x", "--llava", "1.1", "--video_dir_path", str(vids), "--clip_feat_path", str(outd),
                                      "--clip_dir", ck["clip_dir"]])
    mod.main()
    assert sorted(os.listdir(outd)) == ["clip0.pkl", "clip1.pkl", "clip2.pkl", "clip3.pkl"]     # broken.npy: reported, no file
    assert pickle.load(open(outd / "clip1.pkl", "rb")) == "sentinel" and "clip1.npy" not in seen_at_open
    # flush after every 2 processed videos: when the third processed video (clip3) is opened, the first two are on disk
    assert {"clip0.pkl", "clip2.pkl"} <= set(seen_at_open["clip3.npy"])
    from video_chatgpt.eval.model_utils import get_seq_frames
    from video_chatgpt.train import collate_video_features, load_video_features
    csd = {k: v.cuda().bfloat16() for k, v in ck["clip_sd"].items()}
    batch = []
    for name in ("clip0", "clip2", "clip3"):
        f = load_video_features(str(outd), f"{name}.pkl")
        assert isinstance(f, np.ndarray) and f.dtype == np.float16 and f.shape == (356, 1024)
        T = len(clips[name])
        assert (f[T:100] == 0).all() and np.abs(f[:T]).sum() > 0
        # load_video samples min(total, 100) frames at the reference's segment midpoints (eval/model_utils.py:55-79),
        # which repeats / drops frames for short clips: the expectation follows the same indices
        sampled = clips[name][get_seq_frames(T, min(T, 100))]
        hid = O.clip_hidden_states(csd, ck["clip_cfg"], O.preprocess_frames(sampled).cuda().bfloat16(), 2)[-1]
        ref = O.st_pool_numpy(hid[:, 1:].float().cpu().numpy().astype("float16"))
        err = np.linalg.norm(f.astype(np.float32) - ref.astype(np.float32)) / np.linalg.norm(ref.astype(np.float32))
        assert err < 2e-2, (name, err)
        batch.append({"video": f})
    assert collate_video_features(batch).shape == (3, 356, 1024)


@torch.no_grad()
def test_chat_py_caller_sequence(tmp_path):
    """The call sequence of the reference's chat front end (video_chatgpt/chat.py:28-40,137-170) against the
    mirror objects `initialize_model` returns: attribute accesses, fp16 pixel values into the tower,
    hidden_states[-2][:, 1:], pooling, generate(do_sample=True, temperature, stopping_criteria), decode.
    With a vanishing temperature sampling is arg-max, so the text must equal the greedy path's."""
    from PIL import Image
    from _checkpoint import make_tiny_checkpoint
    from video_chatgpt.constants import DEFAULT_VID_END_TOKEN, DEFAULT_VID_START_TOKEN, DEFAULT_VIDEO_PATCH_TOKEN
    from video_chatgpt.eval.model_utils import initialize_model
    from video_chatgpt.inference import get_spatio_temporal_features_torch, video_chatgpt_infer
    from video_chatgpt.model.utils import KeywordsStoppingCriteria
    from video_chatgpt.video_conversation import SeparatorStyle, conv_templates
    ck = make_tiny_checkpoint(tmp_path)
    model, vision_tower, tokenizer, image_processor, video_token_len = initialize_model(ck["model_dir"], max_seq=1024)
    frame_size = (image_processor.crop_size["height"], image_processor.crop_size["width"])
    assert frame_size == (224, 224)
    if model.get_model().vision_config.use_vid_start_end:
        replace_token = DEFAULT_VID_START_TOKEN + DEFAULT_VIDEO_PATCH_TOKEN * video_token_len + DEFAULT_VID_END_TOKEN
    else:
        replace_token = DEFAULT_VIDEO_PATCH_TOKEN * video_token_len
    frames = [Image.fromarray(f) for f in O.make_frames(33, 5)]
    video_tensor = image_processor.preprocess(frames, return_tensors="pt")["pixel_values"]
    state = conv_templates["pg-video-llava"].copy()
    state.append_message(state.roles[0], "w20 w21 w22\n<video>")
    state.append_message(state.roles[1], None)
    prompt = state.get_prompt().replace("<video>", replace_token, 1)
    input_ids = torch.as_tensor(tokenizer([prompt]).input_ids).cuda()
    stop_str = state.sep if state.sep_style != SeparatorStyle.TWO else state.sep2
    stopping_criteria = KeywordsStoppingCriteria([stop_str], tokenizer, input_ids)
    video_tensor = video_tensor.half().cuda()                       # chat.py feeds fp16 pixel values
    image_forward_outs = vision_tower(video_tensor, output_hidden_states=True)
    frame_features = image_forward_outs.hidden_states[-2][:, 1:]
    feats = get_spatio_temporal_features_torch(frame_features)
    with torch.inference_mode():
        output_ids = model.generate(input_ids, video_spatio_temporal_features=feats.unsqueeze(0), do_sample=True,
                                    temperature=1e-4, max_new_tokens=min(8, 1536), stopping_criteria=[stopping_criteria])
    input_token_len = input_ids.shape[1]
    assert (input_ids != output_ids[:, :input_token_len]).sum().item() == 0
    outputs = tokenizer.batch_decode(output_ids[:, input_token_len:], skip_special_tokens=True)[0].strip()
    greedy = video_chatgpt_infer(frames, "w20 w21 w22", "pg-video-llava", model, vision_tower, tokenizer, image_processor,
                                 video_token_len, do_sample=False, max_new_tokens=8)
    print(f"[dropin] chat.py sequence -> {outputs!r}; video_chatgpt_infer (greedy) -> {greedy!r}")
    assert outputs == greedy and len(outputs.split()) >= 1
