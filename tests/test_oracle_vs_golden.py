"""Pins the oracle (oracle/spann3r_oracle.py) to outputs of the REAL reference.

The golden npz files were produced by tools/make_golden.py, which imports /root/reference and runs
`Spann3R.forward` on CPU in strict fp32 with the same synthetic checkpoint / frames.  Tolerance:
2e-5 relative L2 = fp32 reassociation noise between two eager PyTorch programs (SURVEY.md §6 measured
1-3e-6 run-to-run on the reference itself).
"""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, get_state_dict, rel_l2
from oracle import spann3r_oracle as orc
from spann3r_b200 import synth

TOL = 2e-5

CASES = [
    ("cfg1_224_2f_raw.npz", False, 2, 224, 224),
    ("seq_224_4f_sharp.npz", True, 4, 224, 224),
    ("seq_384x512_3f_sharp.npz", True, 3, 384, 512),
]


def _sub_tokens(t, g):
    return t[:, ::int(g["meta/tok_stride"]), ::8]


@pytest.mark.parametrize("fname,sharpen,nf,H,W", CASES)
def test_forward_matches_reference(fname, sharpen, nf, H, W):
    g = np.load(os.path.join(GOLDEN, fname))
    sd = get_state_dict(sharpen)
    frames = synth.make_frames(nf, H, W)
    trace = []
    preds, preds_all, mem = orc.forward(sd, frames, return_memory=True, trace=trace)
    s = int(g["meta/px_stride"])
    worst = 0.0
    for i, p in enumerate(preds):
        for k, v in p.items():
            e = rel_l2(v[:, ::s, ::s], g[f"preds/{i}/{k}"])
            worst = max(worst, e)
            assert e < TOL, (fname, i, k, e)
    for i, (_, r2) in enumerate(preds_all):
        for k, v in r2.items():
            e = rel_l2(v[:, ::s, ::s], g[f"preds_all/{i}/res2/{k}"])
            assert e < TOL, (fname, i, k, e)
    assert rel_l2(_sub_tokens(mem.mem_k, g), g["mem/mem_k_sub"]) < TOL
    assert rel_l2(_sub_tokens(mem.mem_v, g), g["mem/mem_v_sub"]) < TOL
    assert rel_l2(mem.mem_attn, g["mem/mem_attn"]) < 1e-4
    assert np.array_equal(mem.mem_count.numpy(), g["mem/mem_count"])
    # per-stage activations captured by forward hooks in the reference (step 0)
    assert rel_l2(_sub_tokens(trace[0]["feat_k1"], g), g["act/attn_head_1#0"]) < TOL
    assert rel_l2(_sub_tokens(trace[0]["feat_k2"], g), g["act/attn_head_2#0"]) < TOL
    assert rel_l2(_sub_tokens(trace[0]["dec1"][1], g), g["act/dust3r.dec_blocks.0#0"]) < TOL
    assert rel_l2(_sub_tokens(trace[0]["dec2"][1], g), g["act/dust3r.dec_blocks2.0#0"]) < TOL
    assert rel_l2(_sub_tokens(trace[0]["cur_v"], g), g["act/value_out#0"]) < TOL


# BASELINE config 2 itself -- the headline 10-frame 512x384 sequence -- on both checkpoints SURVEY.md §8d names (sharpened =
# headline; raw = ill-conditioned memory reads from the 7th frame on: ~10 surviving weights per row after the 5e-4 cut).
CFG2_CASES = [("cfg2_384x512_10f_sharp.npz", True, 2e-5), ("cfg2_384x512_10f_raw.npz", False, 2e-4)]


@pytest.mark.parametrize("fname,sharpen,tol", CFG2_CASES)
def test_config2_headline_matches_reference(fname, sharpen, tol):
    g = np.load(os.path.join(GOLDEN, fname))
    sd = get_state_dict(sharpen)
    preds, preds_all, mem = orc.forward(sd, synth.make_frames(10, 384, 512), return_memory=True)
    s = int(g["meta/px_stride"])
    worst = 0.0
    for i, p in enumerate(preds):
        assert set(p.keys()) == {k.split("/")[-1] for k in g.files if k.startswith(f"preds/{i}/")}
        for k, v in p.items():
            assert torch.isfinite(v).all()
            worst = max(worst, rel_l2(v[:, ::s, ::s], g[f"preds/{i}/{k}"]))
    for i, (_, r2) in enumerate(preds_all):
        for k, v in r2.items():
            worst = max(worst, rel_l2(v[:, ::s, ::s], g[f"preds_all/{i}/res2/{k}"]))
    print(fname, "worst rel-L2 %.2e" % worst)
    assert worst < tol, worst
    assert mem.mem_k.shape[1] == 9 * 768 and np.array_equal(mem.mem_count.numpy(), g["mem/mem_count"])
    assert rel_l2(mem.mem_attn, g["mem/mem_attn"]) < 10 * tol


# Portrait frames (the landscape wrapper transposes every head output, dust3r/utils/misc.py:66-94) and the
# mem_pos_enc=True constructor variant (RoPE in the value encoder): real-reference runs without activation hooks.
VARIANT_CASES = [
    ("seq_288x224_4f_sharp.npz", 4, 288, 224, False),
    ("seq_512x384_3f_sharp.npz", 3, 512, 384, False),
    ("seq_224_3f_sharp_mempos.npz", 3, 224, 224, True),
]


@pytest.mark.parametrize("fname,nf,H,W,mem_pos_enc", VARIANT_CASES)
def test_portrait_and_mempos_match_reference(fname, nf, H, W, mem_pos_enc):
    g = np.load(os.path.join(GOLDEN, fname))
    sd = get_state_dict(True)
    frames = synth.make_frames(nf, H, W)
    preds, preds_all, mem = orc.forward(sd, frames, return_memory=True, mem_pos_enc=mem_pos_enc)
    s = int(g["meta/px_stride"])
    for i, p in enumerate(preds):
        assert set(p.keys()) == {k.split("/")[-1] for k in g.files if k.startswith(f"preds/{i}/")}
        for k, v in p.items():
            assert v.shape[1:3] == (min(H, W), max(H, W)), (k, v.shape)       # always landscape
            assert rel_l2(v[:, ::s, ::s], g[f"preds/{i}/{k}"]) < TOL, (fname, i, k)
    for i, (_, r2) in enumerate(preds_all):
        for k, v in r2.items():
            assert rel_l2(v[:, ::s, ::s], g[f"preds_all/{i}/res2/{k}"]) < TOL, (fname, i, k)
    assert rel_l2(_sub_tokens(mem.mem_k, g), g["mem/mem_k_sub"]) < TOL
    assert rel_l2(_sub_tokens(mem.mem_v, g), g["mem/mem_v_sub"]) < TOL
    assert rel_l2(mem.mem_attn, g["mem/mem_attn"]) < 1e-4
    assert np.array_equal(mem.mem_count.numpy(), g["mem/mem_count"])


def test_state_dict_spec_counts(spec):
    keys = spec["spann3r"]
    assert len(keys) == 1101  # SURVEY.md §8b
    n_params = sum(int(np.prod(s)) for s in keys.values())
    # 658.7 M distinct parameters + the 8 aliased layerK_rn copies that the state dict lists twice
    assert abs(n_params - 665.3e6) < 0.5e6


def test_rope_matches_curope_formula():
    """oracle rope2d == the loop form of rope_2d_cpu (croco/models/curope/curope.cpp:11-47)."""
    torch.manual_seed(0)
    B, H, N, D = 2, 3, 10, 64
    tok = torch.randn(B, H, N, D)
    pos = torch.randint(0, 32, (B, N, 2))
    out = orc.rope2d(tok, pos)
    exp = tok.clone()
    Q = D // 4
    for half in range(2):
        for q in range(Q):
            inv = 1.0 / (100.0 ** (q / Q))
            ang = pos[:, :, half].float() * inv
            c, s = ang.cos()[:, None, :], ang.sin()[:, None, :]
            u = tok[..., half * 2 * Q + q]
            v = tok[..., half * 2 * Q + q + Q]
            exp[..., half * 2 * Q + q] = u * c - v * s
            exp[..., half * 2 * Q + q + Q] = v * c + u * s
    assert rel_l2(out, exp) < 1e-6


def _pair_graph(forward_fn, frames):
    """The pairwise graph `dust3r.inference.inference` builds for a complete scene graph (every ordered pair once;
    the reference's symmetrised duplicates carry the same numbers)."""
    v1i, v2i, c1, c2 = [], [], [], []
    for a in range(len(frames)):
        for b in range(len(frames)):
            if a == b:
                continue
            r1, r2 = forward_fn(frames[a], frames[b])
            v1i.append(a); v2i.append(b); c1.append(r1["conf"].cpu()); c2.append(r2["conf"].cpu())
    return {"view1": {"idx": v1i}, "view2": {"idx": v2i}, "pred1": {"conf": torch.cat(c1)}, "pred2": {"conf": torch.cat(c2)}}


def test_offline_reconstruction_matches_reference():
    """SURVEY.md §8f rank 2: make_pairs -> inference -> Spann3R.offline_reconstruction of the REAL reference
    (tools/make_golden.py:run_offline) vs the oracle's restatement."""
    g = np.load(os.path.join(GOLDEN, "offline_224_4f_sharp.npz"))
    sd = get_state_dict(True)
    frames = synth.make_frames(4, 224, 224)
    graph = _pair_graph(lambda a, b: orc.dust3r_forward(sd, a, b), frames)
    # the pairwise confidences agree with the reference's inference() output
    for i in range(len(g["graph/view1_idx"])):
        a, b = int(g["graph/view1_idx"][i]), int(g["graph/view2_idx"][i])
        j = [k for k in range(len(graph["view1"]["idx"])) if graph["view1"]["idx"][k] == a and graph["view2"]["idx"][k] == b][0]
        assert rel_l2(graph["pred1"]["conf"][j][::4, ::4], g["graph/pred1_conf"][i]) < TOL
        assert rel_l2(graph["pred2"]["conf"][j][::4, ::4], g["graph/pred2_conf"][i]) < TOL
    preds, preds_all, idx_used = orc.offline_reconstruction(sd, frames, graph)
    assert list(idx_used) == list(g["idx_used"])
    s = int(g["meta/px_stride"])
    for i, p in enumerate(preds):
        for k, v in p.items():
            assert rel_l2(v[:, ::s, ::s], g[f"preds/{i}/{k}"]) < TOL, (i, k)
