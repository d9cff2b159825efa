"""GPU (B200) parity tests — the CUDA path, called through the C ABI (ctypes) and the public Python
mirror, against (a) golden vectors produced by the reference's own code, (b) the CPU oracle on the same
seeded inputs, and (c) size-independent properties at the full 10 s / 48 kHz clip size.

Tolerances (bf16 tensor-core operands, fp32 accumulation and fp32 residual streams; the reference is fp32):
  * single GEMM vs fp32 matmul of the same bf16-rounded operands ............ rel-L2 <= 1e-3
  * attention (bf16 P, bf16 output) ........................................ rel-L2 <= 1e-2
  * one DiT evaluation vs reference ........................................ rel-L2 <= 2e-2
  * codec encode / decode vs oracle ........................................ rel-L2 <= 2e-2 / 3e-2
  * separate() waveforms vs reference (32 evaluations compound) ............ SNR >= 30 dB
  * integer outputs (sizes, lengths, masks, anchors) ....................... bit-exact
"""
import pytest
import torch

from _util import rel_l2, snr_db
from oracle.make_golden import load_samaudio_forward, load_separate, wav_positions

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    import __graft_entry__ as g
    g.build()
    from sam_audio_b200 import _capi
    assert torch.cuda.is_available()
    return _capi


@pytest.mark.parametrize("M,N,K,bn,bk,cg", [
    (128, 256, 64, 256, 64, 1), (300, 256, 256, 256, 64, 1), (1000, 512, 2048, 128, 64, 1),
    (2500, 2048, 2048, 256, 64, 1), (300, 96, 96, 96, 32, 1), (777, 128, 160, 128, 32, 1),
    (500, 192, 192, 192, 64, 1), (333, 96, 192, 96, 64, 1), (129, 64, 128, 64, 64, 1), (1, 256, 64, 256, 64, 1),
    # cta_group::2 pairs (256-row tiles)
    (256, 256, 64, 256, 64, 2), (300, 512, 256, 256, 64, 2), (2500, 2048, 2048, 256, 64, 2),
    (16000, 2816, 2816, 256, 64, 2), (100, 256, 128, 256, 64, 2), (5000, 11008, 512, 256, 64, 0)])
def test_tcgen05_gemm(capi, M, N, K, bn, bk, cg):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N + K)
    a = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    b = torch.randn(N, K, device="cuda", generator=g).bfloat16()
    c = torch.full((M, N), float("nan"), device="cuda")
    capi.check(capi.lib().sab_test_gemm(M, N, K, a.data_ptr(), b.data_ptr(), c.data_ptr(), bn, bk, cg, capi.stream_ptr()))
    torch.cuda.synchronize()
    assert not torch.isnan(c).any()
    assert rel_l2(c, a.float() @ b.float().t()) < 1e-3


@pytest.mark.parametrize("items,heads,Tq,Tk", [(2, 2, 64, 64), (2, 3, 250, 250), (3, 2, 37, 5), (1, 2, 300, 130),
                                               (1, 1, 1, 1), (2, 2, 250, 512)])
def test_attention(capi, items, heads, Tq, Tk):
    g = torch.Generator(device="cuda").manual_seed(Tq + Tk)
    q, k, v = (torch.randn(items * t, heads * 128, device="cuda", generator=g).bfloat16() for t in (Tq, Tk, Tk))
    mask = torch.ones(items, Tk, dtype=torch.uint8, device="cuda")
    for i in range(items):
        mask[i, max(1, Tk - 3 * (i + 1)):] = 0
    o = torch.zeros(items * Tq, heads * 128, device="cuda", dtype=torch.bfloat16)
    capi.check(capi.lib().sab_test_attention(items, heads, Tq, Tk, q.data_ptr(), k.data_ptr(), v.data_ptr(),
                                             mask.data_ptr(), o.data_ptr(), capi.stream_ptr()))
    torch.cuda.synchronize()
    qf, kf, vf = (x.float().view(items, -1, heads, 128).permute(0, 2, 1, 3) for x in (q, k, v))
    s = (qf @ kf.transpose(-1, -2) / 128 ** 0.5).masked_fill(~mask.bool()[:, None, None, :], float("-inf"))
    ref = (torch.softmax(s, -1) @ vf).permute(0, 2, 1, 3).reshape(items * Tq, heads * 128)
    assert rel_l2(o.float(), ref) < 1e-2


@pytest.mark.parametrize("items,heads,T", [(1, 1, 256), (2, 3, 250), (3, 2, 37), (2, 2, 129), (1, 1, 1), (2, 1, 128)])
def test_tcgen05_self_attention(capi, items, heads, T):
    """TMA + tcgen05 QK^T / in-TMEM softmax / TS-form PV kernel (T <= 256) vs fp32 torch, ragged key masks."""
    g = torch.Generator(device="cuda").manual_seed(T + items)
    q, k, v = (torch.randn(items * T, heads * 128, device="cuda", generator=g).bfloat16() for _ in range(3))
    mask = torch.ones(items, T, dtype=torch.uint8, device="cuda")
    for i in range(items):
        mask[i, max(1, T - 3 * (i + 1)):] = 0
    o = torch.zeros(items * T, heads * 128, device="cuda", dtype=torch.bfloat16)
    capi.check(capi.lib().sab_test_attention_tc(items, heads, T, q.data_ptr(), k.data_ptr(), v.data_ptr(),
                                                mask.data_ptr(), o.data_ptr(), 0, 0, capi.stream_ptr()))
    torch.cuda.synchronize()
    qf, kf, vf = (x.float().view(items, T, heads, 128).permute(0, 2, 1, 3) for x in (q, k, v))
    s = (qf @ kf.transpose(-1, -2) / 128 ** 0.5).masked_fill(~mask.bool()[:, None, None, :], float("-inf"))
    ref = (torch.softmax(s, -1) @ vf).permute(0, 2, 1, 3).reshape(items * T, heads * 128)
    assert rel_l2(o.float(), ref) < 1e-2


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("items,heads,T", [(1, 1, 256), (2, 3, 250), (3, 2, 37), (2, 2, 129), (1, 1, 1), (2, 1, 128),
                                           (40, 8, 250), (37, 5, 131)])
def test_tcgen05_self_attention_v2(capi, items, heads, T, exact):
    """Second-generation kernel (attention_tc2.cuh): 16 softmax warps, P/O per key half in TMEM, TMA-stored output;
    exact = two-pass row maximum, otherwise the single-pass softmax with a logit bound (here the Cauchy-Schwarz bound
    of the actual q, k); polynomial exp2 on 3 of 8 pairs.  The last two shapes give every persistent CTA several work
    items (the cross-item pipeline: prefetch, TMEM hand-over, staging-tile hand-over)."""
    g = torch.Generator(device="cuda").manual_seed(T + items)
    q, k, v = (torch.randn(items * T, heads * 128, device="cuda", generator=g).bfloat16() for _ in range(3))
    mask = torch.ones(items, T, dtype=torch.uint8, device="cuda")
    for i in range(items):
        mask[i, max(1, T - 3 * (i % 7 + 1)):] = 0
    o = torch.full((items * T, heads * 128), float("nan"), device="cuda", dtype=torch.bfloat16)
    qn = q.float().view(-1, heads, 128).norm(dim=-1).max()
    kn = k.float().view(-1, heads, 128).norm(dim=-1).max()
    shift = -1.0 if exact else float(qn * kn / 128 ** 0.5 * 1.4426950408889634) + 0.25
    qf, kf, vf = (x.float().view(items, T, heads, 128).permute(0, 2, 1, 3) for x in (q, k, v))
    s = (qf @ kf.transpose(-1, -2) / 128 ** 0.5).masked_fill(~mask.bool()[:, None, None, :], float("-inf"))
    ref = (torch.softmax(s, -1) @ vf).permute(0, 2, 1, 3).reshape(items * T, heads * 128)
    for poly in (3, 0):
        o.fill_(float("nan"))
        capi.check(capi.lib().sab_test_attention_tc2(items, heads, T, q.data_ptr(), k.data_ptr(), v.data_ptr(),
                                                     mask.data_ptr(), o.data_ptr(), shift, poly, None, capi.stream_ptr()))
        torch.cuda.synchronize()
        assert not torch.isnan(o.float()).any()
        assert rel_l2(o.float(), ref) < 1e-2, (poly, exact)
    if not exact:
        # the engine's production variant: log2(e)/sqrt(hd) already folded into q (as the QKV epilogue does), logits
        # bounded by 50 in the log2 domain, p = 2^s with neither scale nor shift (shift_log2 == 0 selects it)
        qs = (q.float() * (1.4426950408889634 / 128 ** 0.5)).bfloat16()
        s2 = (qs.float().view(items, T, heads, 128).permute(0, 2, 1, 3) @ kf.transpose(-1, -2)) * 0.6931471805599453
        assert float(s2.abs().max()) < 50 * 0.6931471805599453
        ref2 = (torch.softmax(s2.masked_fill(~mask.bool()[:, None, None, :], float("-inf")), -1) @ vf)
        ref2 = ref2.permute(0, 2, 1, 3).reshape(items * T, heads * 128)
        o.fill_(float("nan"))
        capi.check(capi.lib().sab_test_attention_tc2(items, heads, T, qs.data_ptr(), k.data_ptr(), v.data_ptr(),
                                                     mask.data_ptr(), o.data_ptr(), 0.0, 3, None, capi.stream_ptr()))
        torch.cuda.synchronize()
        assert not torch.isnan(o.float()).any()
        assert rel_l2(o.float(), ref2) < 1e-2


def test_long_sequence_uses_streaming_attention(tiny_model):
    """T > 256 frames (a 12 s clip) falls back from the single-pass tcgen05 kernel to the streaming one;
    the result must agree with the same clip's first 10 s only in shape/finite-ness (different content),
    and batch invariance must still hold."""
    from sam_audio_b200 import SAMAudioProcessor
    from sam_audio_b200.synthetic import synthetic_clip, synthetic_noise
    proc = SAMAudioProcessor(1920, 48000)
    aud = [synthetic_clip(0, 48000 * 12)]
    noise = synthetic_noise(1, 300).cuda()
    a = tiny_model.separate(proc(descriptions=["thunder"], audios=aud).to("cuda"), noise=noise)
    b = tiny_model.separate(proc(descriptions=["thunder"], audios=aud).to("cuda"), noise=noise)
    assert a.target[0].shape == (48000 * 12,) and torch.isfinite(a.target[0]).all()
    assert torch.equal(a.target[0], b.target[0])


def test_dit_evaluation_vs_reference_golden(tiny_model, golden_dir):
    """SAMAudio.forward (ragged pad mask, text mask, anchors, with and without video) vs the reference's
    own SAMAudio.forward output (tests/golden/samaudio_forward_tiny.pt)."""
    g = load_samaudio_forward(golden_dir)
    for tag, vid in (("video", g["video"]), ("novideo", torch.zeros_like(g["video"]))):
        out = tiny_model.forward(g["noisy"].cuda(), g["feats"].cuda(), g["text"].cuda(), g["time"].cuda(),
                                 masked_video_features=vid.cuda(),
                                 text_mask=g["text_mask"].cuda(), anchor_ids=g["anchor_ids"].cuda(),
                                 anchor_alignment=g["anchor_alignment"].cuda(), audio_pad_mask=g["pad_mask"].cuda())
        assert rel_l2(out.cpu(), g["out"][tag]) < 2e-2, tag


def test_dit_evaluation_none_arguments_vs_reference_golden(tiny_model, golden_dir):
    """The `None` cases of SAMAudio.forward mean what they mean in the reference: no video term (align.py:41-42),
    no anchor term (model.py:57-58), time-only memory (model.py:170-172) — golden = the reference's own output."""
    g = load_samaudio_forward(golden_dir)
    out = tiny_model.forward(g["noisy"].cuda(), g["feats"].cuda(), g["text"].cuda(), g["time"].cuda(),
                             text_mask=g["text_mask"].cuda(), audio_pad_mask=g["pad_mask"].cuda())
    assert rel_l2(out.cpu(), g["out"]["none_video_anchors"]) < 2e-2
    out = tiny_model.forward(g["noisy"].cuda(), g["feats"].cuda(), None, g["time"].cuda(), audio_pad_mask=g["pad_mask"].cuda())
    assert rel_l2(out.cpu(), g["out"]["none_text"]) < 2e-2
    # and they differ from the zeros-video / <null>-anchor path separate() takes
    assert rel_l2(g["out"]["none_video_anchors"], g["out"]["novideo"]) > 1e-3


@pytest.mark.parametrize("L", [1, 8, 12, 20])
def test_dit_evaluation_text_lengths_vs_oracle(tiny_model, tiny_cfg, tiny_sd, L):
    """Cross-attention paths by text length: fused into the cross.wq GEMM epilogue (L <= 8), the small-L kernel
    (L <= 16) and the streaming kernel (L > 16) — each against the CPU oracle on the same inputs."""
    from oracle import restate
    g = torch.Generator().manual_seed(100 + L)
    B, T = 2, 29
    noisy = torch.randn(B, T, 256, generator=g)
    f = torch.randn(B, T, 128, generator=g)
    feats = torch.cat([f, f], 2)
    text = torch.randn(B, L, 768, generator=g)
    tmask = torch.ones(B, L, dtype=torch.bool)
    tmask[1, max(1, L - 2):] = False
    pad = restate.mask_from_sizes(torch.tensor([29.0, 17.0]))
    ids, al = restate.process_anchors(None, pad, 1920, 48000)
    time = torch.tensor([0.25, 0.75])
    ref = restate.samaudio_forward(tiny_sd, tiny_cfg, noisy, feats, text, time, torch.zeros(B, 1024, T), tmask, ids, al, pad)
    out = tiny_model.forward(noisy.cuda(), feats.cuda(), text.cuda(), time.cuda(), text_mask=tmask.cuda(),
                             masked_video_features=torch.zeros(B, 1024, T).cuda(),      # zeros, as separate() passes
                             anchor_ids=ids.cuda(), anchor_alignment=al.cuda(), audio_pad_mask=pad.cuda())
    assert rel_l2(out.cpu(), ref) < 2e-2


@pytest.fixture(scope="module")
def small_model_and_sd():
    """sam-audio-small stand-in (d=1536, 12 layers, 12 heads): production tile shapes, 2-CTA GEMMs, T=250."""
    from sam_audio_b200.config import stand_in_config
    from sam_audio_b200.model import SAMAudio
    from sam_audio_b200.synthetic import make_state_dict
    from sam_audio_b200.text_encoder import SyntheticTextEncoder
    cfg = stand_in_config("sam-audio-small")
    sd = make_state_dict(cfg, seed=1)
    m = SAMAudio(cfg, text_encoder=SyntheticTextEncoder())
    m.load_state_dict(sd)
    return m.eval().cuda(), cfg, sd


def test_dit_evaluation_production_shapes_vs_oracle(small_model_and_sd):
    """One ODE function evaluation at production width and clip length (B=5 x T=250 -> M=1250 rows: cta_group::2 GEMM
    pairs, tcgen05 self-attention, fused text cross-attention) vs the fp32 CPU oracle."""
    from oracle import restate
    m, cfg, sd = small_model_and_sd
    g = torch.Generator().manual_seed(5)
    B, T, L = 5, 250, 3
    noisy = torch.randn(B, T, 256, generator=g)
    f = torch.randn(B, T, 128, generator=g)
    feats = torch.cat([f, f], 2)
    text = torch.randn(B, L, 768, generator=g)
    tmask = torch.ones(B, L, dtype=torch.bool)
    pad = restate.mask_from_sizes(torch.tensor([250.0, 250.0, 199.0, 250.0, 120.0]))
    ids, al = restate.process_anchors([[["+", 1.0, 3.0]], [], [], [["-", 0.0, 9.0]], []], pad, 1920, 48000)
    time = torch.full((B,), 0.40625)
    ref = restate.samaudio_forward(sd, cfg, noisy, feats, text, time, torch.zeros(B, 1024, T), tmask, ids, al, pad)
    out = m.forward(noisy.cuda(), feats.cuda(), text.cuda(), time.cuda(), text_mask=tmask.cuda(),
                    masked_video_features=torch.zeros(B, 1024, T).cuda(),
                    anchor_ids=ids.cuda(), anchor_alignment=al.cuda(), audio_pad_mask=pad.cuda())
    assert rel_l2(out.cpu(), ref) < 2e-2


def test_separate_full_clip_size_vs_oracle(small_model_and_sd):
    """BASELINE clip size end to end (one 10 s @ 48 kHz clip, production-width model): codec encode, 2 midpoint steps
    (4 evaluations; ode_opt is the reference's own knob), codec decode of target + residual, vs the CPU oracle."""
    from oracle import restate
    from sam_audio_b200 import SAMAudioProcessor
    from sam_audio_b200.synthetic import synthetic_clip, synthetic_noise, synthetic_text_features
    m, cfg, sd = small_model_and_sd
    proc = SAMAudioProcessor(1920, 48000)
    aud, desc = [synthetic_clip(3)], ["dog barking"]
    host = proc(descriptions=desc, audios=aud)
    noise = synthetic_noise(1, 250)
    out = m.separate(proc(descriptions=desc, audios=aud).to("cuda"), noise=noise.cuda(),
                     ode_opt={"method": "midpoint", "options": {"step_size": 0.5}})
    tf, tm = synthetic_text_features(desc)
    tgt, res = restate.separate(sd, cfg, host.audios, host.audio_pad_mask, host.sizes, tf, tm, host.anchor_ids,
                                host.anchor_alignment, noise, n_steps=2)
    assert out.target[0].shape == (480000,)
    assert snr_db(out.target[0].cpu(), tgt[0]) > 30.0 and snr_db(out.residual[0].cpu(), res[0]) > 30.0


def test_native_t5_encoder_vs_transformers(capi):
    """sab_t5_forward (tcgen05 GEMMs + relative-bias attention) vs transformers.T5EncoderModel with the same
    random t5-base-shaped weights, ragged descriptions (padding mask) — tolerance as for one DiT evaluation."""
    from sam_audio_b200.config import T5EncoderConfig
    from sam_audio_b200.text_encoder import T5TextEncoder, t5_relative_buckets
    enc = T5TextEncoder(T5EncoderConfig(), allow_random_init=True).cuda()
    texts = ["man speaking", "a dog barking loudly in the distance near a busy street", "thunder", "car honking twice"]
    ours, mask = enc(texts)
    tok = enc.tokenizer(texts, truncation=True, max_length=512, padding="longest", return_tensors="pt")
    ref = enc.model(input_ids=tok["input_ids"].cuda(), attention_mask=tok["attention_mask"].cuda())["last_hidden_state"]
    assert torch.equal(mask.cpu(), tok["attention_mask"].bool()) and ours.shape == ref.shape
    m = mask[..., None].float()
    assert rel_l2(ours * m, ref * m) < 2e-2                 # padded positions carry no information
    # bucket table = transformers' own function
    from transformers.models.t5.modeling_t5 import T5Attention
    L = 40
    rp = torch.arange(L)[None, :] - torch.arange(L)[:, None]
    hf = T5Attention._relative_position_bucket(rp, bidirectional=True, num_buckets=32, max_distance=128)
    tab = t5_relative_buckets(L)
    assert torch.equal(tab[(rp + L - 1)].long(), hf)


def test_codec_vs_oracle(tiny_model, tiny_cfg, tiny_sd):
    from oracle import restate
    from sam_audio_b200.synthetic import synthetic_clip
    wav = torch.stack([synthetic_clip(i, 1920 * 11 + 300) for i in range(3)])      # not a hop multiple -> reflect pad
    ref = restate.codec_encode(tiny_sd, tiny_cfg.audio_codec, wav).transpose(1, 2)
    feats = tiny_model._get_audio_features(wav.cuda())
    assert feats.shape == (3, 12, 256)
    assert torch.equal(feats[:, :, :128], feats[:, :, 128:])                       # model.py:183-184 duplication
    assert rel_l2(feats[:, :, :128].cpu(), ref) < 2e-2
    lat = torch.randn(3, 12, 256, generator=torch.Generator().manual_seed(3))
    ref_w = restate.codec_decode(tiny_sd, tiny_cfg.audio_codec, lat.transpose(1, 2).reshape(6, 128, 12)).view(3, 2, -1)
    out = torch.empty(3, 2, 12 * 1920, device="cuda")
    tiny_model._ensure_engine().decode(lat.cuda(), 3, 12, out)
    torch.cuda.synchronize()
    assert rel_l2(out.cpu(), ref_w) < 3e-2 and float(out.abs().max()) <= 1.0


@pytest.mark.parametrize("cand", [1, 2, 8])
def test_separate_vs_reference_golden(tiny_model, golden_dir, cand):
    """separate() vs the reference's own separate() (candidates 1, 2 and 8: the candidates of a clip share the clip's
    conditioning inside the engine instead of the reference's expand/reshape copies, model.py:193-203)."""
    from sam_audio_b200 import SAMAudioProcessor
    from sam_audio_b200.synthetic import synthetic_clip, synthetic_descriptions
    g = load_separate(golden_dir)
    proc = SAMAudioProcessor(1920, 48000)
    auds = [synthetic_clip(i, n) for i, n in enumerate(g["lens"])]
    batch = proc(descriptions=synthetic_descriptions(2), audios=auds).to("cuda")
    r = g["results"][cand]
    out = tiny_model.separate(batch, noise=r["noise"].cuda(), reranking_candidates=cand)
    assert torch.equal(out.noise.cpu(), r["noise"])
    for ours, ref, n in zip(list(out.target) + list(out.residual), list(r["target"]) + list(r["residual"]),
                            g["wav_lens"] * 2):
        assert ours.shape == (n,)                           # lengths = sizes*1920, bit-exact
        assert snr_db(ours.cpu()[wav_positions(n)], ref) > 30.0
    # every candidate's latent (not only the returned candidate 0) against the reference pipeline's ODE state
    assert rel_l2(tiny_model._last_latent.cpu(), r["latent"]) < 2e-2


def test_decode_small_chunks_equal_unchunked(tiny_model, monkeypatch):
    """Long clips are decoded in chunks of whole clips (target + residual halves of one latent row): forcing the
    smallest chunk (one clip = two waveforms) must reproduce the unchunked decode bit for bit."""
    lat = torch.randn(3, 12, 256, generator=torch.Generator().manual_seed(5)).cuda()
    eng = tiny_model._ensure_engine()
    full = torch.empty(3, 2, 12 * 1920, device="cuda")
    eng.decode(lat, 3, 12, full)
    monkeypatch.setenv("SAB_CODEC_CHUNK_BYTES", "1e6")      # < one waveform's workspace: chunk clamps to one clip
    small = torch.empty_like(full)
    eng.decode(lat, 3, 12, small)
    torch.cuda.synchronize()
    monkeypatch.delenv("SAB_CODEC_CHUNK_BYTES")
    assert torch.equal(full, small)
    assert not torch.equal(small[:, 0], small[:, 1])        # residual is not a copy of the target


def test_candidate_selection_through_attached_rankers_vs_reference_golden(tiny_model, golden_dir):
    """reranking_candidates > 1 with a ranker attached (model.py:306-330): the ranker sees the reference's keyword
    arguments and the returned waveforms are those of each clip's arg-max candidate — golden = the reference's own
    separate() with the same fixed-score stand-in ranker (candidates 1 and 0 win for clips 0 and 1)."""
    from sam_audio_b200 import SAMAudioProcessor
    from sam_audio_b200.ranking import EnsembleRanker
    from sam_audio_b200.synthetic import synthetic_clip, synthetic_descriptions
    g = load_separate(golden_dir)
    r = g["results"]["ranked3"]
    proc = SAMAudioProcessor(1920, 48000)
    auds = [synthetic_clip(i, n) for i, n in enumerate(g["lens"])]
    seen = {}

    class Fixed(torch.nn.Module):
        def forward(self, extracted_audio, input_audio, descriptions, sample_rate):
            seen.update(n=len(extracted_audio), cand=extracted_audio[0].shape[0], inp=input_audio[0].shape,
                        ext=extracted_audio[0].shape, desc=list(descriptions), sr=sample_rate)
            return r["scores"].to(extracted_audio[0].device) * 0.5
    tiny_model.text_ranker = EnsembleRanker([Fixed(), Fixed()], [1.0, 1.0])        # 2 x 0.5 x scores
    try:
        out = tiny_model.separate(proc(descriptions=synthetic_descriptions(2), audios=auds).to("cuda"),
                                  noise=r["noise"].cuda(), reranking_candidates=3)
    finally:
        tiny_model.text_ranker = None
    # input_audio = the (zero-padded) mixture cut at the hop-padded length and expanded over the candidates, as the
    # reference builds it (model.py:317-320): clip 0 is the longest, so its mixture is shorter than the hop-padded output
    assert seen["n"] == 2 and seen["cand"] == 3 and seen["sr"] == 48000
    assert seen["inp"][0] == 3 and seen["inp"][1] == g["lens"][0] <= seen["ext"][1]
    for ours, ref, n in zip(list(out.target) + list(out.residual), list(r["target"]) + list(r["residual"]),
                            g["wav_lens"] * 2):
        assert ours.shape == (n,) and snr_db(ours.cpu()[wav_positions(n)], ref) > 30.0
    # without the ranker candidate 0 is returned: clip 0 differs from the ranked result, clip 1 (winner 0) does not
    plain = tiny_model.separate(proc(descriptions=synthetic_descriptions(2), audios=auds).to("cuda"),
                                noise=r["noise"].cuda(), reranking_candidates=3)
    n0 = g["wav_lens"][0]
    assert snr_db(plain.target[0].cpu()[wav_positions(n0)], r["target"][0]) < 20.0
    assert torch.equal(plain.target[1], out.target[1])


def test_separate_with_anchors_vs_oracle(tiny_model, tiny_cfg, tiny_sd):
    from oracle import restate
    from sam_audio_b200 import SAMAudioProcessor
    from sam_audio_b200.synthetic import (synthetic_clip, synthetic_descriptions, synthetic_noise,
                                          synthetic_text_features)
    proc = SAMAudioProcessor(1920, 48000)
    lens = [7000, 9600, 1921]
    auds = [synthetic_clip(10 + i, n) for i, n in enumerate(lens)]
    anchors = [[["+", 0.02, 0.1]], [["-", 0.0, 0.05], ["+", 0.04, 0.2]], []]
    desc = synthetic_descriptions(3)
    host = proc(descriptions=desc, audios=auds, anchors=anchors)
    noise = synthetic_noise(3, int(host.sizes.max()))
    out = tiny_model.separate(proc(descriptions=desc, audios=auds, anchors=anchors).to("cuda"), noise=noise.cuda())
    tf, tm = synthetic_text_features(desc)
    tgt, res = restate.separate(tiny_sd, tiny_cfg, host.audios, host.audio_pad_mask, host.sizes, tf, tm,
                                host.anchor_ids, host.anchor_alignment, noise)
    for ours, ref in zip(list(out.target) + list(out.residual), tgt + res):
        assert ours.shape == ref.shape and snr_db(ours.cpu(), ref) > 30.0


@pytest.mark.parametrize("method,steps", [("euler", 8), ("rk4", 4), ("midpoint", 5)])
def test_separate_other_fixed_grid_solvers_vs_oracle(tiny_model, tiny_cfg, tiny_sd, method, steps):
    """The reference forwards **ode_opt to torchdiffeq (model.py:285-290): its other fixed-grid solvers — euler and rk4
    (the 3/8 rule) — and other step counts, against the oracle's restatement of the same formulas."""
    from oracle import restate
    from sam_audio_b200 import SAMAudioProcessor
    from sam_audio_b200.synthetic import (synthetic_clip, synthetic_descriptions, synthetic_noise,
                                          synthetic_text_features)
    proc = SAMAudioProcessor(1920, 48000)
    auds = [synthetic_clip(30 + i, n) for i, n in enumerate([9600, 6000])]
    desc = synthetic_descriptions(2)
    host = proc(descriptions=desc, audios=auds)
    noise = synthetic_noise(2, int(host.sizes.max()))
    opt = {"method": method, "options": {"step_size": 1.0 / steps}}
    out = tiny_model.separate(proc(descriptions=desc, audios=auds).to("cuda"), noise=noise.cuda(), ode_opt=opt)
    tf, tm = synthetic_text_features(desc)
    tgt, res, lat = restate.separate(tiny_sd, tiny_cfg, host.audios, host.audio_pad_mask, host.sizes, tf, tm,
                                     host.anchor_ids, host.anchor_alignment, noise, n_steps=steps, method=method,
                                     return_latent=True)
    assert rel_l2(tiny_model._last_latent.cpu(), lat) < 2e-2
    for ours, ref in zip(list(out.target) + list(out.residual), tgt + res):
        assert ours.shape == ref.shape and snr_db(ours.cpu(), ref) > 30.0
    with pytest.raises(NotImplementedError):
        tiny_model.separate(proc(descriptions=desc, audios=auds).to("cuda"), noise=noise.cuda(),
                            ode_opt={"method": "dopri5"})


def test_predict_spans_mutates_batch_but_not_audio(tiny_model):
    """Reference behaviour at the pinned commit (SURVEY App. A.14, model.py:257-268): predicted spans are written into
    the caller's batch (anchor ids / alignment, bit-exact integers) but the audio is that of the un-anchored batch."""
    from types import SimpleNamespace
    from sam_audio_b200 import SAMAudioProcessor
    from sam_audio_b200.synthetic import synthetic_clip, synthetic_noise

    class _Inputs(dict):
        def to(self, device):
            return self

    class _FakeSpanPredictor:                     # stands in for core.audio_visual_encoder.PEAudioFrame
        def __call__(self, input_features, padding_mask, return_spans, **kw):
            assert input_features.shape[-1] == 128 and return_spans
            return SimpleNamespace(spans=[[[0.02, 0.1]], [[0.0, 0.04], [0.06, 0.12]]])

    proc = SAMAudioProcessor(1920, 48000)
    auds = [synthetic_clip(20, 9600), synthetic_clip(21, 7000)]
    noise = synthetic_noise(2, 5).cuda()
    plain = tiny_model.separate(proc(descriptions=["a", "b"], audios=auds).to("cuda"), noise=noise)
    tiny_model.span_predictor = _FakeSpanPredictor()
    tiny_model.span_predictor_transform = lambda text: _Inputs()
    try:
        batch = proc(descriptions=["a", "b"], audios=auds).to("cuda")
        out = tiny_model.separate(batch, noise=noise, predict_spans=True)
    finally:
        tiny_model.span_predictor = None
    ref = proc(descriptions=["a", "b"], audios=auds, anchors=[[["+", 0.02, 0.1]], [["+", 0.0, 0.04], ["+", 0.06, 0.12]]])
    assert torch.equal(batch.anchor_ids.cpu(), ref.anchor_ids) and torch.equal(batch.anchor_alignment.cpu(), ref.anchor_alignment)
    assert all(torch.equal(a, b) for a, b in zip(out.target + out.residual, plain.target + plain.residual))


def test_solver_composition_and_determinism(tiny_model):
    """sab_solve(n_steps=1) == the midpoint formula composed from two sab_dit_forward calls; repeated
    solves are bit-identical (no atomics / nondeterministic reductions on the path)."""
    g = torch.Generator().manual_seed(11)
    B, T, L = 2, 20, 4
    feats = torch.randn(B, T, 128, generator=g)
    feats = torch.cat([feats, feats], 2).cuda()
    text = torch.randn(B, L, 768, generator=g).cuda()
    ids = torch.tensor([[0, 3]] * B).cuda()
    al = torch.zeros(B, T, dtype=torch.long).cuda()
    y0 = torch.randn(B, T, 256, generator=g).cuda()
    eng = tiny_model._ensure_engine()
    tiny_model._install_conditioning(feats, text, None, None, ids, al, None)
    a = torch.empty_like(y0)
    eng.solve(y0, 1, a)
    b = torch.empty_like(y0)
    eng.solve(y0, 1, b)
    assert torch.equal(a, b)
    f0 = torch.empty_like(y0)
    eng.dit_forward(y0, torch.zeros(B, device="cuda"), f0)
    f1 = torch.empty_like(y0)
    eng.dit_forward(y0 + 0.5 * f0, torch.full((B,), 0.5, device="cuda"), f1)
    assert rel_l2(a, y0 + f1) < 5e-3


def test_exact_softmax_fallback_and_many_anchor_ids(tiny_cfg, tiny_sd, golden_dir, monkeypatch):
    """(1) Layers whose QK-norm weights do not bound the logits tightly enough run the exact two-pass softmax variant of
    the tcgen05 attention kernel (forced here through SAB_ATTN_EXACT): same golden as the single-pass path.
    (2) More anchor ids per clip than the plan's initial table (64) rebuild the plan instead of failing."""
    from oracle import restate
    from sam_audio_b200.model import SAMAudio
    from sam_audio_b200.text_encoder import SyntheticTextEncoder
    monkeypatch.setenv("SAB_ATTN_EXACT", "1")
    m = SAMAudio(tiny_cfg, text_encoder=SyntheticTextEncoder())
    m.load_state_dict(tiny_sd)
    m = m.eval().cuda()
    m._ensure_engine()                                     # the env is read when the weights are finalised
    monkeypatch.delenv("SAB_ATTN_EXACT")
    g = load_samaudio_forward(golden_dir)
    out = m.forward(g["noisy"].cuda(), g["feats"].cuda(), g["text"].cuda(), g["time"].cuda(),
                    masked_video_features=g["video"].cuda(), text_mask=g["text_mask"].cuda(),
                    anchor_ids=g["anchor_ids"].cuda(), anchor_alignment=g["anchor_alignment"].cuda(),
                    audio_pad_mask=g["pad_mask"].cuda())
    assert rel_l2(out.cpu(), g["out"]["video"]) < 2e-2
    # 70 anchors on one clip -> 72 ids per row (> 64)
    B, T = 2, 40
    pad = restate.mask_from_sizes(torch.tensor([40.0, 31.0]))
    anchors = [[["+" if i % 2 else "-", 0.01 * i, 0.01 * i + 0.05] for i in range(70)], []]
    ids, al = restate.process_anchors(anchors, pad, 1920, 48000)
    assert ids.shape[1] == 72
    gen = torch.Generator().manual_seed(21)
    noisy = torch.randn(B, T, 256, generator=gen)
    f = torch.randn(B, T, 128, generator=gen)
    feats = torch.cat([f, f], 2)
    text = torch.randn(B, 4, 768, generator=gen)
    time = torch.tensor([0.125, 0.5])
    ref = restate.samaudio_forward(tiny_sd, tiny_cfg, noisy, feats, text, time, torch.zeros(B, 1024, T), None, ids, al, pad)
    out = m.forward(noisy.cuda(), feats.cuda(), text.cuda(), time.cuda(), masked_video_features=torch.zeros(B, 1024, T).cuda(),
                    anchor_ids=ids.cuda(), anchor_alignment=al.cuda(), audio_pad_mask=pad.cuda())
    assert rel_l2(out.cpu(), ref) < 2e-2


def test_missing_or_unknown_weights_fail_loudly(tiny_cfg, tiny_sd):
    from sam_audio_b200.model import SAMAudio
    from sam_audio_b200.text_encoder import SyntheticTextEncoder
    m = SAMAudio(tiny_cfg, text_encoder=SyntheticTextEncoder()).cuda()
    sd = dict(tiny_sd)
    sd.pop("transformer.layers.1.feed_forward.w2.weight")
    m.load_state_dict(sd)
    with pytest.raises(RuntimeError, match="Missing keys"):
        m._ensure_engine()
    m2 = SAMAudio(tiny_cfg, text_encoder=SyntheticTextEncoder()).cuda()
    sd2 = dict(tiny_sd)
    sd2["transformer.bogus.weight"] = torch.zeros(3)
    m2.load_state_dict(sd2)
    with pytest.raises(RuntimeError, match="unexpected weight"):
        m2._ensure_engine()
    # strict=False: the same two defects are reported, not raised (torch's _IncompatibleKeys)
    m4 = SAMAudio(tiny_cfg, text_encoder=SyntheticTextEncoder()).cuda()
    sd4 = dict(sd2)
    sd4.pop("audio_codec.decoder.model.0.bias")
    m4.load_state_dict(sd4, strict=False)
    m4._ensure_engine()
    res = m4._push_weights()
    assert res.unexpected_keys == ["transformer.bogus.weight"] and res.missing_keys == ["audio_codec.decoder.model.0.bias"]
    m3 = SAMAudio(tiny_cfg, text_encoder=SyntheticTextEncoder())
    m3.load_state_dict(tiny_sd)
    with pytest.raises(RuntimeError, match="B200 only"):
        m3._ensure_engine()                                  # still on CPU: no fallback


def test_full_size_properties_10s_clips(tiny_model):
    """BASELINE clip size (10 s @ 48 kHz, T = 250): properties that do not need the (slow) CPU oracle.
      * batch invariance: a clip separated alone == the same clip inside a batch (every op is per-sequence);
      * candidates: duplicated noise rows give identical candidates;
      * outputs are finite, bounded by tanh, and of length sizes*1920 exactly."""
    from sam_audio_b200 import SAMAudioProcessor
    from sam_audio_b200.synthetic import synthetic_clip, synthetic_descriptions, synthetic_noise
    proc = SAMAudioProcessor(1920, 48000)
    auds = [synthetic_clip(i) for i in range(3)]
    desc = synthetic_descriptions(3)
    noise = synthetic_noise(3, 250).cuda()
    full = tiny_model.separate(proc(descriptions=desc, audios=auds).to("cuda"), noise=noise)
    one = tiny_model.separate(proc(descriptions=desc[1:2], audios=auds[1:2]).to("cuda"), noise=noise[1:2])
    assert full.target[1].shape == (480000,) and torch.isfinite(full.target[1]).all()
    assert float(full.target[1].abs().max()) <= 1.0
    assert torch.equal(full.target[1], one.target[0]) and torch.equal(full.residual[1], one.residual[0])
    n2 = noise[:1].repeat_interleave(2, 0)
    c2 = tiny_model.separate(proc(descriptions=desc[:1], audios=auds[:1]).to("cuda"), noise=n2, reranking_candidates=2)
    assert torch.equal(c2.target[0], full.target[0])
