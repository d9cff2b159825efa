"""TEST INFRASTRUCTURE — golden-fixture generator (run in the build container only).

    python -m oracle.make_golden            # writes tests/golden/*.pt

Imports the UNMODIFIED reference (oracle/ref_loader.py), loads the seeded
synthetic state dict (sam_audio_b200/synthetic.py) into the reference's own
modules, runs the reference's own code (DiT.forward, SAMAudio.forward,
SAMAudio.separate control flow, SAMAudioProcessor/Batch) on CPU fp32 and

  1. asserts oracle/restate.py reproduces it (this is what "pins" the oracle), and
  2. stores inputs' seeds + the reference outputs as fixtures, which travel to
     the GPU box where /root/reference does not exist.

Third-party pieces the reference cannot run here (dacvae codec, T5) are replaced
inside the reference pipeline by the restated codec / synthetic text features —
those stages are NOT pinned by these fixtures (see oracle/__init__.py).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_loader, restate  # noqa: E402
from sam_audio_b200 import synthetic  # noqa: E402
from sam_audio_b200.config import stand_in_config  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

# Every fixture stays under 1 MB: seeded random inputs are stored as (shape, seed) plus their first HEAD values, which
# the loaders below check after regenerating them, and separate_tiny.pt keeps one waveform sample in WAV_KEEP.
HEAD = 64
WAV_KEEP = 4
VIDEO_SEED = 8


def rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def wav_positions(n: int) -> torch.Tensor:
    """The positions of an n-sample waveform that separate_tiny.pt stores: a fixed pseudo-random 1/WAV_KEEP of them,
    sorted (numpy's legacy RandomState stream does not change between versions)."""
    return torch.from_numpy(np.sort(np.random.RandomState(n).choice(n, n // WAV_KEEP, replace=False)))


def _seeded_video(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


def _check_head(t, head):
    assert torch.equal(t.flatten()[:HEAD], head), "the seeded generator no longer reproduces this golden input"


def load_samaudio_forward(golden_dir):
    """samaudio_forward_tiny.pt with its video input regenerated from the stored seed."""
    g = torch.load(os.path.join(golden_dir, "samaudio_forward_tiny.pt"))
    g["video"] = _seeded_video(g["video_shape"], g["video_seed"])
    _check_head(g["video"], g["video_head"])
    return g


def load_separate(golden_dir):
    """separate_tiny.pt with each result's noise regenerated from the stored seed.  "target" / "residual" hold each
    clip's waveform at wav_positions(n) only; the full lengths n are in "wav_lens"."""
    g = torch.load(os.path.join(golden_dir, "separate_tiny.pt"))
    for r in g["results"].values():
        bc, t, ch = r["noise_shape"]
        r["noise"] = synthetic.synthetic_noise(bc, t, ch, seed=r["noise_seed"])
        _check_head(r["noise"], r["noise_head"])
    return g


class _RestatedCodec(torch.nn.Module):
    """Stands in for sam_audio.model.codec.DACVAE inside the reference pipeline."""

    def __init__(self, sd, ccfg):
        super().__init__()
        self.sd, self.ccfg = sd, ccfg
        self.sample_rate, self.hop_length = ccfg.sample_rate, ccfg.hop_length

    def forward(self, wav):
        return restate.codec_encode(self.sd, self.ccfg, wav)

    def decode(self, z):
        return restate.codec_decode(self.sd, self.ccfg, z)

    def feature_idx_to_wav_idx(self, idx, sample_rate=None):
        w = idx * self.hop_length * 1.0
        return w.int() if torch.is_tensor(w) else int(w)


class _SyntheticText(torch.nn.Module):
    def forward(self, texts):
        return synthetic.synthetic_text_features(texts)


class FakeClip:
    """Stands in for core.vision_encoder.pe.CLIP (third-party, absent): 12x12 average pooling -> fixed random
    projection -> optional L2 normalisation.  Only the reference's wrapper logic around it is under test."""
    DIM = 32

    def __init__(self):
        self.proj = torch.randn(3 * 12 * 12, self.DIM, generator=torch.Generator().manual_seed(5)) / 20.0

    def encode_image(self, x, normalize=True):
        f = torch.nn.functional.adaptive_avg_pool2d(x.float(), 12).flatten(1) @ self.proj.to(x.device)
        return torch.nn.functional.normalize(f, dim=-1) if normalize else f


def build_reference_pipeline(ref, cfg, sd):
    """SAMAudio.__new__ + attach the reference's own sub-modules (SURVEY Appendix B)."""
    from sam_audio.model import model as ref_model
    from sam_audio.model.align import AlignModalities
    from sam_audio.model.config import TransformerConfig as RefTC
    from sam_audio.model.transformer import DiT
    from dataclasses import asdict

    m = ref_model.SAMAudio.__new__(ref_model.SAMAudio)
    torch.nn.Module.__init__(m)
    tc = cfg.transformer
    m.transformer = DiT(RefTC(**asdict(tc)))
    m.proj = torch.nn.Linear(cfg.in_channels, tc.dim)
    m.align_masked_video = AlignModalities(cfg.vision_encoder.dim, tc.dim)
    m.embed_anchors = ref_model.EmbedAnchors(cfg.num_anchors, cfg.anchor_embedding_dim, tc.dim)
    m.memory_proj = torch.nn.Linear(cfg.text_encoder.dim, tc.dim)
    m.timestep_emb = ref_model.SinusoidalEmbedding(tc.dim)
    m.visual_ranker = m.text_ranker = None
    own = {k: v for k, v in sd.items() if not k.startswith("audio_codec.")}
    missing, unexpected = torch.nn.Module.load_state_dict(m, own, strict=False)
    assert not unexpected, unexpected
    assert not missing, missing
    m.audio_codec = _RestatedCodec(sd, cfg.audio_codec)
    m.text_encoder = _SyntheticText()
    vis = torch.nn.Module()
    vis.dim = cfg.vision_encoder.dim
    m.vision_encoder = vis
    return m.eval()


def main():
    torch.manual_seed(0)
    torch.set_grad_enabled(False)
    os.makedirs(GOLDEN, exist_ok=True)
    ref = ref_loader.load()
    from sam_audio.processor import SAMAudioProcessor

    cfg = stand_in_config("sam-audio-tiny")
    sd = synthetic.make_state_dict(cfg, seed=0)
    model = build_reference_pipeline(ref, cfg, sd)
    tc = cfg.transformer

    # ---------------- processor / anchors (integers, bit-exact) ----------------
    proc = SAMAudioProcessor(audio_hop_length=1920, audio_sampling_rate=48000)
    lens = [24000, 15000, 1920, 1921]
    auds = [torch.randn(2 if i % 2 else 1, n, generator=torch.Generator().manual_seed(50 + i))
            for i, n in enumerate(lens)]
    anchors = [[["+", 0.1, 0.3]], [["-", 0.0, 0.11], ["+", 0.05, 0.2]], [], [["+", 0.0, 0.04]]]
    desc = synthetic.synthetic_descriptions(len(lens))
    pg = {"lens": lens, "anchors": anchors, "cases": {}}
    for tag, anc in (("none", None), ("spans", anchors)):
        b = proc(descriptions=desc, audios=auds, anchors=anc)
        o_aud, o_ws = restate.batch_audio(auds)
        o_sizes = restate.wav_to_feature_idx(o_ws, 1920)
        o_mask = restate.mask_from_sizes(o_sizes)
        o_ids, o_al = restate.process_anchors(anc, o_mask, 1920, 48000)
        assert torch.equal(b.audios, o_aud) and torch.equal(b.wav_sizes, o_ws)
        assert torch.equal(b.sizes, o_sizes) and b.sizes.dtype == o_sizes.dtype
        assert torch.equal(b.audio_pad_mask, o_mask)
        assert torch.equal(b.anchor_ids, o_ids) and torch.equal(b.anchor_alignment, o_al)
        pg["cases"][tag] = dict(sizes=b.sizes, wav_sizes=b.wav_sizes, audio_pad_mask=b.audio_pad_mask,
                                anchor_ids=b.anchor_ids, anchor_alignment=b.anchor_alignment,
                                audios_sum=b.audios.double().sum(-1))
    # the survey's measured example: ["+",6.3,7.0] -> frames [158,175)
    b = proc(descriptions=["x"], audios=[torch.zeros(1, 480000)], anchors=[[["+", 6.3, 7.0]]])
    nz = (b.anchor_alignment[0] == 2).nonzero().flatten()
    assert int(nz[0]) == 158 and int(nz[-1]) == 174
    pg["survey_example"] = dict(anchor_alignment=b.anchor_alignment, anchor_ids=b.anchor_ids)
    # masked-video inputs as tensors (reference processor.py:131-155 tensor branch, :197-204): one frame per latent
    # frame picked by linspace().round(), masked pixels zeroed
    gv = torch.Generator().manual_seed(77)
    vids = [torch.randint(0, 256, (n, 3, 4, 6), generator=gv, dtype=torch.uint8) for n in (30, 7, 1, 5)]
    msks = [torch.randint(0, 2, (n, 1, 4, 6), generator=gv, dtype=torch.uint8) for n in (30, 7, 1, 5)]
    masked = proc.mask_videos(vids, msks)
    bv = proc(descriptions=desc, audios=auds, masked_videos=masked)
    pg["video"] = dict(video_lens=[30, 7, 1, 5], masked=[m.clone() for m in masked],
                       frames=[f.clone() for f in bv.masked_video])
    torch.save(pg, os.path.join(GOLDEN, "processor.pt"))
    print("processor: restatement bit-exact vs reference")
    if "--processor-only" in sys.argv:
        return

    # ---------------- DiT.forward + SAMAudio.forward (ragged, anchors) ----------------
    g = torch.Generator().manual_seed(7)
    B, T, L = 3, 37, 5
    sizes = torch.tensor([37.0, 23.0, 30.0])
    pad_mask = restate.mask_from_sizes(sizes)
    x = torch.randn(B, T, tc.dim, generator=g)
    time = torch.tensor([0.0, 0.40625, 0.96875])
    memory = torch.randn(B, L, tc.dim, generator=g)
    mem_mask = torch.tensor([[1, 1, 1, 1, 1], [1, 1, 0, 0, 0], [1, 1, 1, 1, 0]], dtype=torch.bool)
    ref_out = model.transformer(x, time, padding_mask=pad_mask, memory=memory, memory_padding_mask=mem_mask)
    our = restate.dit_forward(sd, tc, x, time, pad_mask, memory, mem_mask)
    e = rel_l2(our, ref_out)
    print(f"DiT.forward restatement vs reference: rel_l2={e:.3e}")
    assert e < 2e-5, e
    torch.save(dict(seed=7, B=B, T=T, L=L, sizes=sizes, time=time, mem_mask=mem_mask, out=ref_out,
                    x=x, memory=memory), os.path.join(GOLDEN, "dit_forward_tiny.pt"))

    noisy = torch.randn(B, T, 256, generator=g)
    feats = torch.randn(B, T, 128, generator=g)
    feats = torch.cat([feats, feats], 2)
    text = torch.randn(B, L, 768, generator=g)
    video = _seeded_video((B, 1024, T), VIDEO_SEED)
    anc = [[["+", 0.1, 0.5]], [["-", 0.0, 0.2], ["+", 0.1, 0.9]], []]
    ids, al = restate.process_anchors(anc, pad_mask, 1920, 48000)
    outs = {}
    for tag, vid in (("video", video), ("novideo", torch.zeros_like(video))):
        r = model.forward(noisy, feats, text, time, masked_video_features=vid, text_mask=mem_mask,
                          anchor_ids=ids, anchor_alignment=al, audio_pad_mask=pad_mask)
        o = restate.samaudio_forward(sd, cfg, noisy, feats, text, time, vid, mem_mask, ids, al, pad_mask)
        e = rel_l2(o, r)
        print(f"SAMAudio.forward[{tag}] restatement vs reference: rel_l2={e:.3e}")
        assert e < 2e-5, e
        outs[tag] = r
    # the three `None` cases of SAMAudio.forward (no video term / no anchor term / time-only memory)
    for tag, kw in (("none_video_anchors", dict(text_features=text, text_mask=mem_mask)),
                    ("none_text", dict(text_features=None, text_mask=None))):
        r = model.forward(noisy, feats, kw["text_features"], time, masked_video_features=None,
                          text_mask=kw["text_mask"], anchor_ids=None, anchor_alignment=None, audio_pad_mask=pad_mask)
        o = restate.samaudio_forward(sd, cfg, noisy, feats, kw["text_features"], time, None, kw["text_mask"], None, None,
                                     pad_mask)
        e = rel_l2(o, r)
        print(f"SAMAudio.forward[{tag}] restatement vs reference: rel_l2={e:.3e}")
        assert e < 2e-5, e
        outs[tag] = r
    torch.save(dict(noisy=noisy, feats=feats, text=text, video_shape=tuple(video.shape), video_seed=VIDEO_SEED,
                    video_head=video.flatten()[:HEAD].clone(), time=time, text_mask=mem_mask,
                    anchor_ids=ids, anchor_alignment=al, pad_mask=pad_mask, out=outs),
               os.path.join(GOLDEN, "samaudio_forward_tiny.pt"))

    # ---------------- visual prompting: PerceptionEncoder transform + chunked encode (reference classes) ----------------
    from sam_audio.model import vision_encoder as ref_ve
    from sam_audio.model.config import PerceptionEncoderConfig as RefPEC
    fake = FakeClip()
    ref_ve.pe.CLIP = type("CLIP", (), {"from_config": staticmethod(lambda name: fake)})   # the third-party tower: a stand-in
    enc = ref_ve.PerceptionEncoder(RefPEC(dim=FakeClip.DIM))
    gv2 = torch.Generator().manual_seed(78)
    vids = [torch.randint(0, 256, (n, 3, 20, 28), generator=gv2, dtype=torch.uint8) for n in (310, 7, 1)]
    feats = enc(vids)                                             # 310 frames > batch_size 300: two chunks; zero-padded
    o = restate.vision_encode(vids, lambda x: fake.encode_image(x, normalize=True), 336, 300)
    assert feats.shape == (3, 310, FakeClip.DIM) and rel_l2(o, feats) < 1e-4, rel_l2(o, feats)
    big = torch.randint(0, 256, (2, 3, 360, 640), generator=gv2, dtype=torch.uint8)
    tb = enc.transform(big)                                       # the reference's own torchvision transform
    lvl = ((tb * 0.5 + 0.5) * 255).round().to(torch.uint8)
    mine = restate.frame_transform(big)
    mis = float((((mine * 0.5 + 0.5) * 255).round().to(torch.uint8) != lvl).float().mean())
    print(f"vision: chunked encode ok; frame transform vs torchvision: {mis:.2e} of the uint8 levels differ (by 1)")
    assert mis < 1e-4
    torch.save(dict(video_lens=[310, 7, 1], seed=78, feats=feats, big_levels=lvl, proj=fake.proj),
               os.path.join(GOLDEN, "vision.pt"))

    # ---------------- separate(): control flow, candidates, unbatch ----------------
    lens2 = [24000, 15000]
    auds2 = [synthetic.synthetic_clip(i, n) for i, n in enumerate(lens2)]
    desc2 = synthetic.synthetic_descriptions(2)
    sep = {}

    def stored(r, noise, seed, **extra):
        return dict(target=[t[wav_positions(t.numel())].clone() for t in r.target],
                    residual=[t[wav_positions(t.numel())].clone() for t in r.residual], noise_shape=tuple(noise.shape),
                    noise_seed=seed, noise_head=noise.flatten()[:HEAD].clone(), **extra)
    for cand in (1, 2, 8):
        batch = proc(descriptions=desc2, audios=auds2)
        Tn = int(batch.sizes.max())
        noise = synthetic.synthetic_noise(2 * cand, Tn, seed=4321)
        r = model.separate(batch, noise=noise, reranking_candidates=cand)
        tf, tm = synthetic.synthetic_text_features(desc2)
        tgt, res, lat = restate.separate(sd, cfg, batch.audios, batch.audio_pad_mask, batch.sizes, tf, tm,
                                         batch.anchor_ids, batch.anchor_alignment, noise,
                                         candidates=cand, return_latent=True)
        for a, b_ in zip(tgt + res, list(r.target) + list(r.residual)):
            assert a.shape == b_.shape, (a.shape, b_.shape)
            e = rel_l2(a, b_)
            assert e < 1e-4, e
        print(f"separate(candidates={cand}) restatement vs reference pipeline: ok "
              f"(lens {[t.numel() for t in r.target]})")
        sep[cand] = stored(r, noise, 4321, latent=lat)
    # candidate selection through an attached text ranker (model.py:316-328): a stand-in with fixed scores — the
    # call-site logic (argument shapes, argmax, which candidate's waveforms are returned) is the reference's
    class _FixedRanker(torch.nn.Module):
        SCORES = torch.tensor([[0.1, 0.9, 0.3], [0.7, 0.2, 0.4]])

        def forward(self, extracted_audio, input_audio, descriptions, sample_rate):
            assert len(extracted_audio) == 2 and extracted_audio[0].shape[0] == 3 and input_audio[0].shape[0] == 3
            assert input_audio[1].shape[-1] == extracted_audio[1].shape[-1] and sample_rate == 48000
            return self.SCORES.clone()
    model.text_ranker = _FixedRanker()
    batch = proc(descriptions=desc2, audios=auds2)
    noise = synthetic.synthetic_noise(2 * 3, int(batch.sizes.max()), seed=777)
    r = model.separate(batch, noise=noise, reranking_candidates=3)
    model.text_ranker = None
    sep["ranked3"] = stored(r, noise, 777, scores=_FixedRanker.SCORES.clone())
    torch.save(dict(lens=lens2, wav_lens=[t.numel() for t in r.target], results=sep),
               os.path.join(GOLDEN, "separate_tiny.pt"))
    for f in sorted(os.listdir(GOLDEN)):
        print(f, os.path.getsize(os.path.join(GOLDEN, f)))


if __name__ == "__main__":
    main()
