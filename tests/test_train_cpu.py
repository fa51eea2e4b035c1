"""CPU tests of the training-mode host logic (spann3r_b200/train.py, _recompute.py).

`_recompute.py` is what the BACKWARD pass of training mode differentiates (PyTorch recompute of each engine stage); the
forward always runs the CUDA library.  Here the restatements are pinned, stage by stage, to the oracle (itself pinned to the
real reference), and the autograd plumbing of `train._Stage` is checked with a stand-in for the native call."""
import numpy as np
import pytest
import torch

from conftest import get_state_dict, rel_l2
from oracle import spann3r_oracle as orc
from spann3r_b200 import _recompute as R
from spann3r_b200 import synth, train

H, W = 64, 96


@pytest.fixture(scope="module")
def sd():
    return get_state_dict(True)


def test_recompute_stages_equal_the_oracle(sd):
    torch.manual_seed(0)
    fr = synth.make_frames(2, H, W)
    img = torch.cat([f["img"] for f in fr])
    with torch.no_grad():
        feats = R.encode(sd, img)
        ref, pos = orc.encode_image(sd, img)
        assert rel_l2(feats, ref) < 1e-5
        f1, f2 = ref[:1], ref[1:]
        fuse = f1 + 0.1 * torch.randn_like(f1)
        k1, k2, pts, conf = R.step(sd, fuse, f1, f2, H, W)
        d1, d2 = orc.decoder(sd, fuse, pos[:1], f2, pos[1:])
        assert rel_l2(k1, orc.key_head(sd, 1, f1, d1[-1])) < 1e-5 and rel_l2(k2, orc.key_head(sd, 2, f2, d2[-1])) < 1e-5
        r1 = orc.dpt_head(sd, "dust3r.downstream_head1", d1, H, W)
        r2 = orc.dpt_head(sd, "dust3r.downstream_head2", d2, H, W)
        assert rel_l2(pts[0], r1["pts3d"]) < 1e-5 and rel_l2(conf[1], r2["conf"]) < 1e-5 and rel_l2(pts[1], r2["pts3d"]) < 1e-5
        for rope in (False, True):
            v = R.value(sd, r1["pts3d"], k1, rope)
            assert rel_l2(v, orc.encode_cur_value(sd, r1["pts3d"], mem_pos_enc=rope) + k1) < 1e-5
        # training-mode read: attn_thresh = 0 (no cut, no renormalisation), optional dropout keep-scale
        om = orc.SpatialMemory(sd, attn_thresh=0)
        g = torch.Generator().manual_seed(3)
        ks = [torch.randn(1, 24, 1024, generator=g) for _ in range(2)]
        vs = [torch.randn(1, 24, 1024, generator=g) for _ in range(2)]
        for k, v in zip(ks, vs):
            om.add_mem(k, v)
        q = torch.randn(1, 24, 1024, generator=g)
        assert rel_l2(R.memory_read(sd, q, torch.cat(ks, 1), torch.cat(vs, 1)), om.memory_read(q)) < 1e-5


def test_stage_function_backward_is_autograd_of_the_recompute():
    """train._Stage: forward = the 'native' callable (no graph), backward = autograd of the torch restatement -> the
    gradients must equal plain autograd through the restatement (activations AND parameters, unused ones None)."""
    torch.manual_seed(1)
    names = ["w", "b", "unused"]
    params = [torch.randn(5, 7, requires_grad=True), torch.randn(5, requires_grad=True), torch.randn(3, requires_grad=True)]
    x = torch.randn(4, 7, requires_grad=True)

    def torch_fn(P, a):
        y = torch.tanh(a @ P["w"].t() + P["b"])
        return y, y.sum(dim=1)

    calls = []

    def native(a):
        calls.append(a.requires_grad)
        return tuple(t.detach() for t in torch_fn(dict(zip(names, params)), a))

    y, s = train._apply(native, torch_fn, names, params, x)
    assert calls == [True] or calls == [False]
    loss = (y * torch.arange(5.0)).sum() + (s ** 2).sum()
    loss.backward()
    got = [x.grad.clone()] + [p.grad.clone() if p.grad is not None else None for p in params]
    x.grad = None
    for p in params:
        p.grad = None
    y2, s2 = torch_fn(dict(zip(names, params)), x)
    ((y2 * torch.arange(5.0)).sum() + (s2 ** 2).sum()).backward()
    assert torch.allclose(got[0], x.grad, atol=1e-6)
    assert torch.allclose(got[1], params[0].grad, atol=1e-6) and torch.allclose(got[2], params[1].grad, atol=1e-6)
    assert got[3] is None and params[2].grad is None


def test_stage_parameter_partition_covers_every_key_once(spec):
    """Every parameter belongs to exactly one stage Function (else it would get no / a double gradient)."""
    from spann3r_b200 import Spann3R
    m = Spann3R(dus3r_name=None)
    seen = {}
    for stage in ("encode", "memread", "step", "value"):
        names, params = train.stage_params(m, stage)
        assert len(names) == len(set(names)) and len(names) == len(params)
        for n in names:
            assert n not in seen, (n, stage, seen.get(n))
            seen[n] = stage
    every = [n for n, _ in m.named_parameters(remove_duplicate=False)]
    missing = sorted(set(every) - set(seen))
    assert missing == ["dust3r.mask_token"], missing        # unused by the forward path (dust3r/model.py: masking is off)
    assert all(p.requires_grad for p in m.parameters())     # trainable by default, like the reference's modules


def philox_keep_scale_numpy(seed: int, n: int, p: float) -> np.ndarray:
    """Host restatement of csrc/memory.cu:dropout_scale (Philox4x32-10, counter = idx / 4, key = seed)."""
    idx = np.arange(n, dtype=np.uint64)
    c = idx >> np.uint64(2)
    ctr = [(c & np.uint64(0xFFFFFFFF)).astype(np.uint64), (c >> np.uint64(32)).astype(np.uint64),
           np.zeros(n, np.uint64), np.zeros(n, np.uint64)]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    M0, M1, MASK = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = M0 * ctr[0], M1 * ctr[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & MASK, p1 >> np.uint64(32), p1 & MASK
        ctr = [hi1 ^ ctr[1] ^ k0, lo1, hi0 ^ ctr[3] ^ k1, lo0]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & MASK, (k1 + np.uint64(0xBB67AE85)) & MASK
    words = np.stack(ctr, axis=1)[np.arange(n), (idx & np.uint64(3)).astype(np.int64)]
    u = (words >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    return np.where(u >= np.float32(p), np.float32(1.0 / (1.0 - p)), np.float32(0.0)).astype(np.float32)


def test_philox_host_restatement_statistics():
    ks = philox_keep_scale_numpy(1234567890123, 200000, 0.15)
    keep = (ks > 0).mean()
    assert abs(keep - 0.85) < 0.004 and np.allclose(ks[ks > 0], 1 / 0.85)
    assert not np.array_equal(ks, philox_keep_scale_numpy(1234567890124, 200000, 0.15))
    # known answer of Philox4x32-10 (Random123 kat_vectors: counter 0, key 0)
    z = np.zeros(1, np.uint64)
    ctr, k0, k1 = [z.copy(), z.copy(), z.copy(), z.copy()], np.uint64(0), np.uint64(0)
    M0, M1, MASK = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = M0 * ctr[0], M1 * ctr[2]
        ctr = [(p1 >> np.uint64(32)) ^ ctr[1] ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ ctr[3] ^ k1, p0 & MASK]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & MASK, (k1 + np.uint64(0xBB67AE85)) & MASK
    assert [int(v[0]) for v in ctr] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]


class _TorchEngine:
    """Stand-in for engine.Engine on the CPU: every 'native' stage evaluates the recompute restatement (no graph, like the CUDA
    library), so `train.forward_train` + `train._Stage` run end to end without a GPU."""

    def __init__(self, sd, B, H, W):
        self.P, self.B, self.H, self.W = sd, B, H, W
        self.N = (H // 16) * (W // 16)
        self.max_images, self.device = 16, torch.device("cpu")
        self.bank_k, self.bank_v = [], []

    def encode(self, img):
        return R.encode(self.P, img)

    def decode(self, f_fuse, f2, want_all=False):
        self._dec_in = (f_fuse, f2)

    def keyheads(self, f1, f2):
        k1, k2, self._pts, self._conf = R.step(self.P, self._dec_in[0], f1, self._dec_in[1], self.H, self.W)
        return k1, k2

    def heads(self):
        return self._pts, self._conf

    def value(self, pts3d, k1, transposed=False, rope=False):
        return R.value(self.P, pts3d, k1, rope)

    def memory_append(self, bank, k, v):
        self.bank_k.append(k)
        self.bank_v.append(v)
        bank.len += self.N

    def memory_read(self, bank, feat, thresh, drop_p=0.0, seed=0):
        assert thresh == 0.0 and drop_p == 0.0
        return R.memory_read(self.P, feat, torch.cat(self.bank_k, 1), torch.cat(self.bank_v, 1))


def test_training_forward_and_recompute_backward_end_to_end_on_cpu(monkeypatch, sd):
    """`train.forward_train` (the real frame loop, stage Functions and parameter routing) over a torch stand-in engine:
    outputs equal the oracle's training-branch forward and the gradients equal autograd through the oracle.
    (On the GPU the same backward is fed by the CUDA forward, whose activations differ by <= 3e-4: tests/test_train_gpu.py.)
    Both sides run in float64: in fp32 their gradients differ by 2e-4 .. 4e-4 depending on the host's CPU kernels and
    thread count, rounding noise of the same size as the bound; in float64 they agree to ~1e-15."""
    from spann3r_b200 import Spann3R
    import spann3r_b200.engine as E

    class _Bank:
        def __init__(self, batch, cap, device):
            self.len, self.cap = 0, cap
    monkeypatch.setattr(E, "MemoryBank", _Bank)
    sd = {k: v.double() for k, v in sd.items()}
    m = Spann3R(dus3r_name=None, memory_dropout=0.0).double()
    m.load_state_dict(sd, strict=True)
    m.train()
    P = dict(m.named_parameters(remove_duplicate=False))
    eng = _TorchEngine({k: v.detach() for k, v in P.items()}, 1, H, W)
    monkeypatch.setattr(m, "_engine_for", lambda *a, **k: eng)
    monkeypatch.setattr(m, "_dev", lambda t: t)
    frames = [{"img": f["img"].double()} for f in synth.make_frames(3, H, W)]
    g = torch.Generator().manual_seed(5)
    wts = [torch.randn(1, H, W, 3, generator=g, dtype=torch.float64) for _ in range(3)]

    def loss_of(preds):
        tot = 0.0
        for p, w in zip(preds, wts):
            k = "pts3d" if "pts3d" in p else "pts3d_in_other_view"
            tot = tot + (p[k] * w).sum() + 0.1 * p["conf"].log().sum()
        return tot

    watch = ["dust3r.enc_blocks.3.attn.qkv.weight", "dust3r.dec_blocks.7.cross_attn.projk.weight", "attn_head_2.0.weight",
             "norm_k.weight", "value_encoder.4.mlp.fc2.weight", "value_out.bias",
             "dust3r.downstream_head1.dpt.scratch.refinenet2.resConfUnit1.conv1.weight", "pos_patch_embed.proj.weight"]
    preds, _ = m(frames)
    loss = loss_of(preds)
    loss.backward()
    got = {k: P[k].grad.clone() for k in watch}
    sdr = {k: v.clone().requires_grad_(k in watch) for k, v in sd.items()}
    ref, _ = orc.forward.__wrapped__(sdr, frames, attn_thresh=0, sim_thresh=1.0)
    for p, r in zip(preds, ref):
        for k in r:
            assert rel_l2(p[k].detach(), r[k].detach()) < 1e-5, k
    grads = torch.autograd.grad(loss_of(ref), [sdr[k] for k in watch])
    errs = {k: rel_l2(got[k], gr) for k, gr in zip(watch, grads)}
    assert all(got[k].dtype == torch.float64 for k in watch)
    assert max(errs.values()) < 2e-4, errs
