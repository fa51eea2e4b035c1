#!/usr/bin/env python
"""Generate the committed golden vectors by running the REAL reference (CPU, strict fp32).

Runs only in the authoring container (needs /root/reference, which does not exist on the
GPU box).  Nothing under tests/, bench.py or smoke() imports this file; they read the small
fixtures it writes into tests/golden/.

    python tools/make_golden.py            # everything (~10 min on 8 cores)
    python tools/make_golden.py --only spec

Outputs
  spann3r_b200/state_dict_spec.json   key -> shape of the reference Spann3R state dict
  tests/golden/cfg1_224_2f_raw.npz    BASELINE config 1 (2 x 224x224), raw random-init weights, outputs (::3, ::3)
  tests/golden/seq_224_4f_sharp.npz   4 x 224x224, sharpened weights (two memory reads), outputs (::3, ::3)
  tests/golden/seq_384x512_3f_sharp.npz  3 x 384x512, sharpened, outputs sub-sampled (::12, ::12), tokens ::21
  tests/golden/offline_224_4f_sharp.npz  offline mode: 4 x 224x224, complete pair graph -> offline_reconstruction, outputs (::3, ::3)
  tests/golden/seq_288x224_4f_sharp.npz  PORTRAIT 4 x (H=288, W=224): transpose_to_landscape (dust3r/utils/misc.py:66-94), outputs (::6, ::6)
  tests/golden/seq_512x384_3f_sharp.npz  PORTRAIT 3 x (H=512, W=384), outputs sub-sampled (::12, ::12)
  tests/golden/seq_224_3f_sharp_mempos.npz  3 x 224x224 with Spann3R(mem_pos_enc=True) (RoPE inside the value encoder), outputs (::6, ::6)
  tests/golden/cfg2_384x512_10f_sharp.npz  BASELINE config 2 exactly (10 x 384x512, sharpened ckpt), outputs (::16, ::16), tokens ::21   [--only cfg2]
  tests/golden/cfg2_384x512_10f_raw.npz    the same on the RAW random-init checkpoint (SURVEY 8d: report both)                           [--only cfg2]
Each npz also holds sub-sampled per-stage activations (first call of each hooked module) captured with forward hooks
so that a parity failure can be localised to a stage.

Every file stays under 1 MB.  Output maps are sub-sampled with a pixel stride (`meta/px_stride`) of at most the
16-pixel patch, so every patch contributes samples; memory keys / values and token activations keep every
`meta/tok_stride`-th token and every 8th channel.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
sys.path.insert(0, REPO)
GOLD = os.path.join(REPO, "tests", "golden")


def build_reference(seed=0, sharpen=False, mem_pos_enc=False):
    sys.path.insert(0, REF)
    torch.serialization.add_safe_globals([argparse.Namespace])
    from spann3r.model import Spann3R  # noqa  (reference)
    from spann3r_b200 import synth

    spec_path = os.path.join(REPO, "spann3r_b200", "state_dict_spec.json")
    tmp = "/tmp/fake_dust3r.pth"
    if not os.path.exists(spec_path):
        # bootstrap: build once with whatever init to learn the key inventory
        from dust3r.model import AsymmetricCroCo3DStereo  # noqa
        inf = float("inf")  # noqa
        net = eval(synth.DUST3R_ARGS.replace("ManyAR_PatchEmbed", "PatchEmbedDust3R"))
        torch.save({"args": argparse.Namespace(model=synth.DUST3R_ARGS), "model": net.state_dict()}, tmp)
        m = Spann3R(dus3r_name=tmp, use_feat=False)
        spec = {"spann3r": {k: list(v.shape) for k, v in m.state_dict().items()},
                "reference_commit": "f89d6a23", "torch": torch.__version__}
        with open(spec_path, "w") as f:
            json.dump(spec, f, indent=0)
        print("wrote", spec_path, len(spec["spann3r"]), "keys")
    spec = synth.load_spec(spec_path)
    dust3r_sd = synth.make_state_dict(spec, seed=seed, prefix="dust3r.")
    torch.save({"args": argparse.Namespace(model=synth.DUST3R_ARGS), "model": dust3r_sd}, tmp)
    t0 = time.time()
    m = Spann3R(dus3r_name=tmp, use_feat=False, mem_pos_enc=mem_pos_enc)
    sd = synth.make_state_dict(spec, seed=seed, sharpen=sharpen)
    missing = m.load_state_dict(sd, strict=True)
    print("reference built in %.1fs" % (time.time() - t0), missing)
    return m.eval()


def sub(t, tok_stride=7, ch_stride=8):
    t = t.detach().float()
    if t.ndim == 3:      # [B, N, C] tokens
        return t[:, ::tok_stride, ::ch_stride].contiguous().numpy()
    if t.ndim == 4:      # [B, C, H, W] feature map
        return t[:, ::ch_stride, ::9, ::9].contiguous().numpy()
    return t.numpy()


def run(model, frames, out_path, px_stride=1, tok_stride=7, hooks=True):
    acts = {}
    handles = []
    if hooks:
        watch = {
            "dust3r.patch_embed": lambda o: o[0],
            "dust3r.enc_blocks.0": lambda o: o,
            "dust3r.enc_blocks.23": lambda o: o,
            "dust3r.enc_norm": lambda o: o,
            "dust3r.decoder_embed": lambda o: o,
            "dust3r.dec_blocks.0": lambda o: o[0],
            "dust3r.dec_blocks2.0": lambda o: o[0],
            "dust3r.dec_blocks.11": lambda o: o[0],
            "dust3r.dec_blocks2.11": lambda o: o[0],
            "attn_head_1": lambda o: o,
            "attn_head_2": lambda o: o,
            "dust3r.downstream_head1.dpt.act_postprocess.0": lambda o: o,
            "dust3r.downstream_head1.dpt.act_postprocess.3": lambda o: o,
            "dust3r.downstream_head1.dpt.scratch.refinenet4": lambda o: o,
            "dust3r.downstream_head1.dpt.scratch.refinenet1": lambda o: o,
            "dust3r.downstream_head1.dpt": lambda o: o,
            "pos_patch_embed": lambda o: o[0],
            "value_encoder.5": lambda o: o,
            "value_out": lambda o: o,
        }
        mods = dict(model.named_modules())
        for name, pick in watch.items():
            def mk(name, pick):
                def hook(_m, _i, o):
                    k = "act/" + name + "#0"
                    if k not in acts:
                        acts[k] = sub(pick(o), tok_stride=tok_stride)
                return hook
            handles.append(mods[name].register_forward_hook(mk(name, pick)))
    t0 = time.time()
    with torch.no_grad():
        preds, preds_all, mem = model(frames, return_memory=True)
    dt = time.time() - t0
    for h in handles:
        h.remove()
    out = {}
    s = px_stride
    for i, p in enumerate(preds):
        for k, v in p.items():
            out[f"preds/{i}/{k}"] = v[:, ::s, ::s].contiguous().numpy()
    for i, (r1, r2) in enumerate(preds_all):
        for k, v in r2.items():
            out[f"preds_all/{i}/res2/{k}"] = v[:, ::s, ::s].contiguous().numpy()
    out["mem/mem_k_sub"] = sub(mem.mem_k, tok_stride=tok_stride)
    out["mem/mem_v_sub"] = sub(mem.mem_v, tok_stride=tok_stride)
    out["mem/mem_attn"] = mem.mem_attn.numpy()
    out["mem/mem_count"] = mem.mem_count.numpy()
    out["meta/px_stride"] = np.array(s)
    out["meta/tok_stride"] = np.array(tok_stride)
    out["meta/ref_seconds"] = np.array(dt)
    out["meta/threads"] = np.array(torch.get_num_threads())
    finite = all(np.isfinite(v).all() for k, v in out.items() if k.startswith("preds"))
    out.update(acts)
    np.savez_compressed(out_path, **out)
    print(f"wrote {out_path}: {dt:.1f}s ref forward, finite={finite}, "
          f"|pts3d| max {max(np.abs(v).max() for k, v in out.items() if 'pts3d' in k):.3g}, "
          f"{os.path.getsize(out_path)/1e6:.2f} MB")


def run_offline(model, frames, out_path, px_stride=3):
    """demo.py:104-118 offline branch: make_pairs (complete, symmetrized) -> dust3r.inference.inference -> offline_reconstruction."""
    from dust3r.image_pairs import make_pairs  # noqa (reference)
    from dust3r.inference import inference  # noqa (reference)
    imgs_all = [dict(img=f["img"], true_shape=torch.tensor(f["img"].shape[2:]).unsqueeze(0), idx=j, instance=str(j))
                for j, f in enumerate(frames)]
    pairs = make_pairs(imgs_all, scene_graph="complete", prefilter=None, symmetrize=True)
    t0 = time.time()
    with torch.no_grad():
        output = inference(pairs, model.dust3r, "cpu", batch_size=2, verbose=False)
        preds, preds_all, idx_used = model.offline_reconstruction(frames, output)
    out = {"idx_used": np.array(idx_used), "graph/view1_idx": np.array(output["view1"]["idx"]),
           "graph/view2_idx": np.array(output["view2"]["idx"]),
           "graph/pred1_conf": output["pred1"]["conf"][:, ::4, ::4].contiguous().numpy(),
           "graph/pred2_conf": output["pred2"]["conf"][:, ::4, ::4].contiguous().numpy(),
           "meta/ref_seconds": np.array(time.time() - t0), "meta/px_stride": np.array(px_stride)}
    s = px_stride
    for i, p in enumerate(preds):
        for k, v in p.items():
            out[f"preds/{i}/{k}"] = v[:, ::s, ::s].contiguous().numpy()
    np.savez_compressed(out_path, **out)
    print(f"wrote {out_path}: idx_used={idx_used}, {time.time() - t0:.1f}s, {os.path.getsize(out_path)/1e6:.2f} MB")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="all")
    args = ap.parse_args()
    from spann3r_b200 import synth
    torch.backends.cuda.matmul.allow_tf32 = False
    os.makedirs(GOLD, exist_ok=True)
    if args.only in ("all", "spec", "cfg1"):
        m = build_reference(sharpen=False)
        if args.only != "spec":
            run(m, synth.make_frames(2, 224, 224), os.path.join(GOLD, "cfg1_224_2f_raw.npz"), px_stride=3)
        del m
    if args.only in ("all", "mempos"):
        m = build_reference(sharpen=True, mem_pos_enc=True)
        run(m, synth.make_frames(3, 224, 224), os.path.join(GOLD, "seq_224_3f_sharp_mempos.npz"), px_stride=6, hooks=False)
        del m
    if args.only in ("all", "cfg2"):   # the headline config itself, both checkpoints (~10 CPU-minutes each on 8 cores)
        for sharpen, tag in ((True, "sharp"), (False, "raw")):
            m = build_reference(sharpen=sharpen)
            # px 16 = one sample per patch: with stride 8, ten frames plus the memory would not fit in 1 MB
            run(m, synth.make_frames(10, 384, 512), os.path.join(GOLD, f"cfg2_384x512_10f_{tag}.npz"), px_stride=16,
                tok_stride=21, hooks=False)
            del m
    if args.only in ("all", "seq224", "seq512", "offline", "portrait"):
        m = build_reference(sharpen=True)
        if args.only in ("all", "portrait"):
            run(m, synth.make_frames(4, 288, 224), os.path.join(GOLD, "seq_288x224_4f_sharp.npz"), px_stride=6, hooks=False)
            run(m, synth.make_frames(3, 512, 384), os.path.join(GOLD, "seq_512x384_3f_sharp.npz"), px_stride=12, hooks=False)
        if args.only in ("all", "offline"):
            run_offline(m, synth.make_frames(4, 224, 224), os.path.join(GOLD, "offline_224_4f_sharp.npz"))
        if args.only in ("all", "seq224"):
            run(m, synth.make_frames(4, 224, 224), os.path.join(GOLD, "seq_224_4f_sharp.npz"), px_stride=3)
        if args.only in ("all", "seq512"):
            run(m, synth.make_frames(3, 384, 512), os.path.join(GOLD, "seq_384x512_3f_sharp.npz"), px_stride=12, tok_stride=21)


if __name__ == "__main__":
    main()
