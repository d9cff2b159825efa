"""CPU: the oracle restatement (oracle/restate.py) against the golden vectors produced by the
reference's own code (oracle/make_golden.py).  This is what pins the oracle."""
import os

import torch

from oracle import restate
from oracle.make_golden import load_samaudio_forward, load_separate, wav_positions
from sam_audio_b200 import synthetic
from _util import rel_l2

torch.set_grad_enabled(False)


def test_dit_forward_matches_reference_golden(golden_dir, tiny_cfg, tiny_sd):
    g = torch.load(os.path.join(golden_dir, "dit_forward_tiny.pt"))
    pad = restate.mask_from_sizes(g["sizes"])
    out = restate.dit_forward(tiny_sd, tiny_cfg.transformer, g["x"], g["time"], pad, g["memory"], g["mem_mask"])
    assert rel_l2(out, g["out"]) < 2e-5


def test_samaudio_forward_matches_reference_golden(golden_dir, tiny_cfg, tiny_sd):
    g = load_samaudio_forward(golden_dir)
    for tag, vid in (("video", g["video"]), ("novideo", torch.zeros_like(g["video"]))):
        out = restate.samaudio_forward(tiny_sd, tiny_cfg, g["noisy"], g["feats"], g["text"], g["time"], vid,
                                       g["text_mask"], g["anchor_ids"], g["anchor_alignment"], g["pad_mask"])
        assert rel_l2(out, g["out"][tag]) < 2e-5, tag
    # the reference's `None` arguments: no video term, no anchor term, time-only memory (model.py:57-58,170-172)
    out = restate.samaudio_forward(tiny_sd, tiny_cfg, g["noisy"], g["feats"], g["text"], g["time"], None,
                                   g["text_mask"], None, None, g["pad_mask"])
    assert rel_l2(out, g["out"]["none_video_anchors"]) < 2e-5
    out = restate.samaudio_forward(tiny_sd, tiny_cfg, g["noisy"], g["feats"], None, g["time"], None, None, None, None,
                                   g["pad_mask"])
    assert rel_l2(out, g["out"]["none_text"]) < 2e-5


def test_processor_restatement_matches_reference_golden(golden_dir):
    g = torch.load(os.path.join(golden_dir, "processor.pt"))
    auds = [torch.randn(2 if i % 2 else 1, n, generator=torch.Generator().manual_seed(50 + i))
            for i, n in enumerate(g["lens"])]
    for tag, anc in (("none", None), ("spans", g["anchors"])):
        ref = g["cases"][tag]
        aud, ws = restate.batch_audio(auds)
        sizes = restate.wav_to_feature_idx(ws, 1920)
        mask = restate.mask_from_sizes(sizes)
        ids, al = restate.process_anchors(anc, mask, 1920, 48000)
        assert torch.equal(ws, ref["wav_sizes"]) and torch.equal(sizes, ref["sizes"])
        assert sizes.dtype == ref["sizes"].dtype == torch.float32
        assert torch.equal(mask, ref["audio_pad_mask"])
        assert torch.equal(ids, ref["anchor_ids"]) and torch.equal(al, ref["anchor_alignment"])
        assert torch.allclose(aud.double().sum(-1), ref["audios_sum"])


def test_midpoint_solver_is_32_evaluations_at_exact_times():
    seen = []

    def f(t, y):
        seen.append(float(t))
        return -y
    y = restate.odeint_midpoint(f, torch.ones(3), 16)
    assert len(seen) == 32
    assert seen == [k / 32 for k in range(32)]            # multiples of 1/32, exact in fp32
    assert abs(float(y[0]) - (1 - 1 / 16 + 0.5 / 256) ** 16) < 1e-6


def test_other_fixed_grid_solvers_orders_of_accuracy():
    """euler / rk4 restatements (torchdiffeq fixed-grid formulas): exact discrete solutions of y' = -y."""
    import math
    f = lambda t, y: -y
    y0 = torch.ones(2, dtype=torch.float64)
    assert abs(float(restate.odeint_fixed(f, y0, 8, "euler")[0]) - (1 - 1 / 8) ** 8) < 1e-12
    h = 1 / 4
    step = 1 - h + h ** 2 / 2 - h ** 3 / 6 + h ** 4 / 24          # any 4th-order RK on a linear ODE
    assert abs(float(restate.odeint_fixed(f, y0, 4, "rk4")[0]) - step ** 4) < 1e-12
    assert abs(float(restate.odeint_fixed(f, y0, 4, "rk4")[0]) - math.exp(-1)) < 1e-4
    assert torch.equal(restate.odeint_fixed(f, y0, 5, "midpoint"), restate.odeint_midpoint(f, y0, 5))


def test_separate_control_flow_matches_reference_golden(golden_dir, tiny_cfg, tiny_sd):
    """encode -> 32 evaluations -> decode -> unbatch, candidates 1 and 8 (reference pipeline output)."""
    g = load_separate(golden_dir)
    auds = [synthetic.synthetic_clip(i, n) for i, n in enumerate(g["lens"])]
    aud, ws = restate.batch_audio(auds)
    sizes = restate.wav_to_feature_idx(ws, 1920)
    mask = restate.mask_from_sizes(sizes)
    ids, al = restate.process_anchors(None, mask, 1920, 48000)
    tf, tm = synthetic.synthetic_text_features(synthetic.synthetic_descriptions(2))
    for cand in (1, 8):                                   # 8 = BASELINE config 4's reranking_candidates
        r = g["results"][cand]
        tgt, res, lat = restate.separate(tiny_sd, tiny_cfg, aud, mask, sizes, tf, tm, ids, al, r["noise"],
                                         candidates=cand, return_latent=True)
        assert lat.shape[0] == 2 * cand and rel_l2(lat, r["latent"]) < 1e-4
        for a, b, n in zip(tgt + res, list(r["target"]) + list(r["residual"]), g["wav_lens"] * 2):
            assert a.shape == (n,) and rel_l2(a[wav_positions(n)], b) < 1e-4


def test_ranked_candidate_selection_matches_reference_golden(golden_dir, tiny_cfg, tiny_sd):
    """model.py:306-330 with an attached (stand-in, fixed-score) text ranker: arg-max candidate per clip."""
    g = load_separate(golden_dir)
    r = g["results"]["ranked3"]
    auds = [synthetic.synthetic_clip(i, n) for i, n in enumerate(g["lens"])]
    aud, ws = restate.batch_audio(auds)
    sizes = restate.wav_to_feature_idx(ws, 1920)
    mask = restate.mask_from_sizes(sizes)
    ids, al = restate.process_anchors(None, mask, 1920, 48000)
    tf, tm = synthetic.synthetic_text_features(synthetic.synthetic_descriptions(2))
    tgt, res = restate.separate(tiny_sd, tiny_cfg, aud, mask, sizes, tf, tm, ids, al, r["noise"], candidates=3,
                                ranker_scores=r["scores"])
    assert r["scores"].argmax(1).tolist() == [1, 0]
    for a, b, n in zip(tgt + res, list(r["target"]) + list(r["residual"]), g["wav_lens"] * 2):
        assert a.shape == (n,) and rel_l2(a[wav_positions(n)], b) < 1e-4


def test_codec_shapes_and_hop(tiny_cfg, tiny_sd):
    cc = tiny_cfg.audio_codec
    assert cc.hop_length == 1920
    wav = synthetic.synthetic_clip(0, 1920 * 3 + 7)[None]
    z = restate.codec_encode(tiny_sd, cc, wav)
    assert z.shape == (1, 128, 4)                         # reflect-padded to 4 frames (codec.py:72-78)
    w = restate.codec_decode(tiny_sd, cc, z)
    assert w.shape == (1, 1, 4 * 1920) and float(w.abs().max()) <= 1.0
