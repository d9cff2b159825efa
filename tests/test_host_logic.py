"""CPU: host-side logic of the drop-in mirror (config, weight-norm folding, synthetic shapes, sharding)."""
import math

import pytest
import torch

from sam_audio_b200.config import SAMAudioConfig, TransformerConfig, stand_in_config
from sam_audio_b200.model import DFLT_ODE_OPT, fold_weight_norm
from sam_audio_b200.parallel import shard_range
from sam_audio_b200.synthetic import codec_param_shapes, make_state_dict


def test_reference_defaults():
    c = SAMAudioConfig()
    t = c.transformer
    assert (t.dim, t.n_heads, t.n_layers, t.head_dim) == (2048, 16, 16, 128)
    assert t.ffn_hidden == 5504 and t.rope_theta == 20000.0        # transformer.py:179-185, :405-406
    assert c.audio_codec.hop_length == 1920 and c.in_channels == 768
    assert DFLT_ODE_OPT == {"method": "midpoint", "options": {"step_size": 2 / 32}}
    assert stand_in_config("sam-audio-large").transformer.ffn_hidden == 7552


def test_config_roundtrip_uses_reference_json_keys():
    c = SAMAudioConfig(transformer={"dim": 1536, "n_heads": 12, "n_layers": 12, "context_dim": 1536})
    d = c.to_dict()
    assert set(d) == {"in_channels", "audio_codec", "text_encoder", "vision_encoder", "transformer", "num_anchors",
                      "anchor_embedding_dim", "visual_ranker", "text_ranker", "span_predictor"}
    c2 = SAMAudioConfig(**d)
    assert c2.transformer.dim == 1536 and c2.audio_codec.encoder_rates == [2, 8, 10, 12]


def test_unsupported_variants_fail_loudly():
    with pytest.raises(NotImplementedError):
        TransformerConfig(dim=1024, n_heads=16).check_supported()        # head_dim 64
    with pytest.raises(NotImplementedError):
        TransformerConfig(non_linearity="gelu").check_supported()
    TransformerConfig().check_supported()


def test_fold_weight_norm_both_spellings():
    g, v = torch.rand(4, 1, 1) + 0.5, torch.randn(4, 3, 7)
    w = g * v / v.flatten(1).norm(dim=1).view(4, 1, 1)
    a = fold_weight_norm({"x.weight_g": g, "x.weight_v": v, "x.bias": torch.zeros(4)})
    b = fold_weight_norm({"x.parametrizations.weight.original0": g, "x.parametrizations.weight.original1": v})
    assert torch.allclose(a["x.weight"], w) and torch.allclose(b["x.weight"], w) and "x.bias" in a
    ref = torch.nn.utils.parametrizations.weight_norm(torch.nn.Conv1d(3, 4, 7))
    sd = ref.state_dict()
    assert torch.allclose(fold_weight_norm(sd)["weight"], ref.weight, atol=1e-6)


def test_synthetic_state_dict_names_and_shapes():
    cfg = stand_in_config("sam-audio-tiny")
    sd = make_state_dict(cfg, seed=0)
    d, hid = 256, cfg.transformer.ffn_hidden
    assert sd["transformer.layers.1.feed_forward.w1.weight"].shape == (hid, d)
    assert sd["transformer.x_embedder.block.block2.project.weight"].shape == (d, d, 3)
    assert sd["transformer.t_block.weight"].shape == (6 * d, d)
    assert sd["proj.weight"].shape == (d, 768)
    assert sd["audio_codec.decoder.model.1.block.1.weight"].shape == (1536, 768, 24)
    assert sd["audio_codec.encoder.block.4.block.4.weight"].shape == (1024, 512, 24)
    assert sd["audio_codec.quantizer.in_proj.weight"].shape == (256, 1024, 1)
    n_codec = sum(math.prod(s) for _, s, _ in codec_param_shapes(cfg.audio_codec))
    assert 60e6 < n_codec < 120e6
    sd2 = make_state_dict(cfg, seed=0)
    assert all(torch.equal(sd[k], sd2[k]) for k in sd)               # deterministic across calls


def test_shard_range_covers_everything_once():
    for n in (0, 1, 7, 8, 256):
        for w in (1, 2, 3, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def test_from_pretrained_local_directory_and_no_cpu_path(tmp_path):
    """The reference's loading contract (base.py:17-62): a directory with config.json + checkpoint.pt; constructor
    overrides are taken from config keys; encoder / ranker keys in the checkpoint are skipped (model.py:346-359);
    weight-normed codec tensors are folded.  Without a GPU the model refuses to run instead of falling back."""
    import json
    from sam_audio_b200 import SAMAudio, SAMAudioProcessor
    from sam_audio_b200.text_encoder import SyntheticTextEncoder
    cfg = stand_in_config("sam-audio-tiny")
    sd = make_state_dict(cfg, seed=0)
    # store one codec conv in weight-norm form and add keys the reference ignores
    w = sd.pop("audio_codec.encoder.block.0.weight")
    sd["audio_codec.encoder.block.0.weight_v"] = 3.0 * w
    sd["audio_codec.encoder.block.0.weight_g"] = w.flatten(1).norm(dim=1).view(-1, 1, 1)
    sd["text_encoder.model.shared.weight"] = torch.zeros(4, 4)
    sd["span_predictor.anything"] = torch.zeros(1)
    (tmp_path / "config.json").write_text(json.dumps(cfg.to_dict()))
    torch.save(sd, tmp_path / "checkpoint.pt")

    m = SAMAudio.from_pretrained(str(tmp_path), text_encoder=SyntheticTextEncoder())
    assert m.cfg.transformer.dim == cfg.transformer.dim and m.sample_rate == 48000
    assert not any(k.startswith(("text_encoder.", "span_predictor.")) for k in m._state)
    assert torch.allclose(m._state["audio_codec.encoder.block.0.weight"], w, atol=1e-6)
    proc = SAMAudioProcessor.from_pretrained(str(tmp_path))
    assert proc.audio_hop_length == 1920 and proc.audio_sampling_rate == 48000
    batch = proc(descriptions=["thunder"], audios=[torch.zeros(1, 4000)])
    with pytest.raises(RuntimeError, match="B200 only"):
        m.eval().separate(batch)


def test_t5_bucket_table_matches_transformers_and_hash_tokenizer_is_stable():
    """Host side of the native T5 path: the relative-position bucket table handed to sab_t5_forward is transformers'
    own bucketing (same fp32 expression, so boundaries round identically), for every length up to the 512-token cap."""
    from transformers.models.t5.modeling_t5 import T5Attention
    from sam_audio_b200.text_encoder import _HashTokenizer, t5_relative_buckets
    for L in (1, 2, 9, 40, 129, 512):
        rp = torch.arange(L)[None, :] - torch.arange(L)[:, None]           # key - query
        hf = T5Attention._relative_position_bucket(rp, bidirectional=True, num_buckets=32, max_distance=128)
        tab = t5_relative_buckets(L)
        assert tab.shape == (2 * L - 1,) and tab.dtype == torch.int32
        assert torch.equal(tab[rp + L - 1].long(), hf)
    tok = _HashTokenizer()
    a = tok(["man speaking", "a dog barking loudly"])
    b = tok(["man speaking", "a dog barking loudly"])
    assert torch.equal(a["input_ids"], b["input_ids"]) and torch.equal(a["attention_mask"], b["attention_mask"])
    assert a["input_ids"].shape == (2, 5) and a["input_ids"][0, 2] == 1 and a["input_ids"][0, 3] == 0   # </s>, then pad
    assert a["attention_mask"].sum(1).tolist() == [3, 5]


def test_separate_validates_ode_opt_before_touching_the_gpu():
    """ode_opt is the reference's pass-through to torchdiffeq (model.py:285-290): fixed-grid methods only, and a
    step_size that divides [0, 1]; the checks run before the engine (and thus a GPU) is needed."""
    from sam_audio_b200.model import SAMAudio
    from sam_audio_b200.text_encoder import SyntheticTextEncoder
    m = SAMAudio(stand_in_config("sam-audio-tiny"), text_encoder=SyntheticTextEncoder())
    for bad in ({"method": "dopri5"}, {"method": "midpoint"}, {"method": "rk4", "options": {"step_size": 0.3}}):
        with pytest.raises(NotImplementedError):
            m.separate(None, ode_opt=bad)
    with pytest.raises(RuntimeError, match="B200 only|no weights"):      # valid options: next stop is the (absent) engine
        m.separate(None, ode_opt={"method": "euler", "options": {"step_size": 0.125}})


def test_from_pretrained_routes_hub_kwargs(tmp_path, monkeypatch):
    """Hub keyword arguments (token, cache_dir, revision, ...) go to snapshot_download, config keys override the
    config, everything else reaches the constructor (reference base.py:17-61 via ModelHubMixin)."""
    import json
    import huggingface_hub
    from sam_audio_b200.model import SAMAudio
    from sam_audio_b200.synthetic import make_state_dict
    from sam_audio_b200.text_encoder import SyntheticTextEncoder
    cfg = stand_in_config("sam-audio-tiny")
    (tmp_path / "config.json").write_text(json.dumps(cfg.to_dict()))
    torch.save(make_state_dict(cfg, seed=0), tmp_path / "checkpoint.pt")
    seen = {}

    def fake_download(repo_id, **kw):
        seen.update(repo_id=repo_id, **kw)
        return str(tmp_path)
    monkeypatch.setattr(huggingface_hub, "snapshot_download", fake_download)
    m = SAMAudio.from_pretrained("facebook/sam-audio-large", token="t0k", cache_dir="/c", revision="r1", num_anchors=3,
                                 text_encoder=SyntheticTextEncoder())
    assert seen == {"repo_id": "facebook/sam-audio-large", "token": "t0k", "cache_dir": "/c", "revision": "r1"}
    assert isinstance(m.text_encoder, SyntheticTextEncoder) and m._state is not None
    res = m.load_state_dict(m._state, strict=False)          # no engine yet: nothing to report
    assert list(res.missing_keys) == [] and list(res.unexpected_keys) == []


def test_perception_encoder_wrapper_host_behaviour():
    from sam_audio_b200.config import PerceptionEncoderConfig
    from sam_audio_b200.vision_encoder import PerceptionEncoder
    enc = PerceptionEncoder(PerceptionEncoderConfig())
    assert enc.batch_size == 300 and enc.image_size == 336 and enc.dim == 1024
    with pytest.raises(RuntimeError, match="B200 only"):
        enc.transform(torch.zeros(2, 3, 8, 8, dtype=torch.uint8))            # no CPU path
    with pytest.raises(NotImplementedError):
        enc.transform(torch.zeros(2, 3, 8, 8))                               # the reference feeds uint8 frames
    with pytest.raises(NotImplementedError):
        enc.encode(torch.zeros(1, 3, 336, 336))                              # no tower attached
    with pytest.raises(NotImplementedError):
        PerceptionEncoder(PerceptionEncoderConfig(interpolation_mode="BILINEAR"))


def test_ensemble_ranker_is_the_weighted_sum():
    from sam_audio_b200.ranking import EnsembleRanker, Ranker

    class A(Ranker):
        def forward(self, **kw):
            return torch.tensor([[1.0, 2.0], [3.0, 4.0]]) * kw["k"]

    class B(Ranker):
        def forward(self, **kw):
            return torch.tensor([[0.5, 0.0], [0.0, 0.5]])
    out = EnsembleRanker([A(), B()], [2.0, 4.0])(k=1.0)
    assert torch.equal(out, torch.tensor([[4.0, 4.0], [6.0, 10.0]]))
    with pytest.raises(TypeError):
        Ranker()                                   # abstract, as the reference's


def test_bench_parity_gate_logic():
    """bench.py's parity gate (BASELINE.md 3.5): passes on small deviations, withholds on a wrong result."""
    import bench
    g = torch.Generator().manual_seed(0)
    cpu = dict(features=torch.randn(1, 10, 128, generator=g), velocity=torch.randn(1, 10, 256, generator=g),
               latent=torch.randn(1, 10, 256, generator=g), wav=torch.randn(2, 1000, generator=g))
    near = {k: v * (1 + 2e-3) for k, v in cpu.items()}
    r = bench.parity_gate(near, cpu)
    assert r["ok"] and abs(r["velocity_rel_l2"] - 2e-3) < 1e-4 and 53 < r["wav_snr_db"] < 55 and r["snr_db"] == r["wav_snr_db"]
    bad = dict(near, wav=cpu["wav"] + 0.1 * torch.randn(2, 1000, generator=g))
    assert not bench.parity_gate(bad, cpu)["ok"]
    bad = dict(near, velocity=-cpu["velocity"])
    assert not bench.parity_gate(bad, cpu)["ok"]


def test_bench_output_dump_is_bounded_and_repeatable(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 .npy files within the byte budget; an array over its share keeps the same
    seeded sample of columns in every row and in every run; small arrays are written whole."""
    import numpy as np
    import bench
    from sam_audio_b200.model import SeparationResult
    monkeypatch.setattr(bench, "DUMP_BYTES", 60_000)
    B, S = 4, 48_000
    wav = torch.arange(B * S, dtype=torch.float32).view(B, S)          # value = row * S + column
    res = SeparationResult(target=list(wav), residual=list(-wav), noise=torch.randn(B, 5, 8).double())
    for run in ("a", "b"):
        bench.write_outputs(bench.sample_outputs(bench.step_outputs(res)), str(tmp_path / run))
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["noise.npy", "residual.npy", "target.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 60_000 + 3 * 128
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    assert all(v.dtype == np.float32 for v in a.values())
    assert all(np.array_equal(v, np.load(tmp_path / "b" / f)) for f, v in a.items())
    t = a["target.npy"]
    cols = t[0]
    assert t.shape == (B, 20_000 // (4 * B)) and (np.diff(cols) > 0).all()
    assert np.array_equal(t, cols[None] + S * np.arange(B, dtype=np.float32)[:, None])
    assert np.array_equal(a["residual.npy"], -t)
    assert np.array_equal(a["noise.npy"], res.noise.float().view(B, -1).numpy())
    g = bench.sample_outputs(bench.step_outputs(torch.stack([wav, -wav], 1)))    # the N > 1 form: [N*B, 2, samples]
    assert sorted(g) == ["residual", "target"] and torch.equal(g["residual"], -g["target"])
    assert g["target"].shape == (B, 30_000 // (4 * B))
