"""Variable-length scoring on the GPU: right-padded batches with per-utterance frame counts against the oracle run on
every utterance at its own length; padding never leaks; lengths == T is bit-identical to the fixed-length path.

Tolerances as elsewhere: <= 1e-4 relative in fp32, <= 2e-2 in bf16 (fp32 state), against the fp64 oracle, per slice
(oracle/compare.py): every utterance, and every 8-frame chunk of it, against its own magnitude."""
import numpy as np
import pytest
import torch

import bimamba_b200 as bm
from oracle import bimamba_oracle as orc
from oracle import compare as cmp
from oracle.varlen_oracle import backend_varlen_ref

pytestmark = pytest.mark.gpu

TOL = cmp.TOL
# shorter than the conv width, around the 8-step checkpoint and 16-step chunk boundaries, and the full padded length
LENGTHS = [1, 2, 3, 7, 8, 9, 15, 16, 17, 40]


def _mamba(d_model, seed):
    p64 = orc.init_mamba_params(d_model, 16, seed=seed, dtype=torch.float64)
    m = bm.Mamba(d_model, 16).cuda()
    m.load_state_dict({k: v.float() for k, v in p64.items()}, strict=True)
    return m, {k: v.float().double().cuda() for k, v in p64.items()}


def _backend(n_layers=2, seed=30):
    layers = [orc.init_encoder_params(144, 16, seed=seed + i) for i in range(n_layers)]
    head = orc.init_head_params(144, seed=seed)
    net = bm.BiMambaBackend(144, n_layers, 16).cuda().eval()
    sd = {f"backbone_layers.{i}.{k}": v for i, p in enumerate(layers) for k, v in p.items()}
    sd.update(head)
    net.load_state_dict(sd, strict=True)
    return net, [{k: v.double().cuda() for k, v in p.items()} for p in layers], {k: v.double().cuda() for k, v in head.items()}


def _autocast(dtype):
    return torch.autocast("cuda", dtype=dtype, enabled=dtype != torch.float32)


def _check_block(m, pr, x, lengths, out, tol):
    for n in sorted(set(lengths)):
        idx = [b for b, v in enumerate(lengths) if v == n]
        ref = orc.bimamba_ref(pr, x[idx, :n].double().cuda())
        cmp.check(f"out(n={n})", out[idx, :n], ref, tol, cmp.frames())


@pytest.mark.parametrize("variant", [1, 3])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("d_model,reps", [(144, 1), (80, 1), (144, 13)])
@pytest.mark.parametrize("sequenced", [False, True])
def test_block_varlen_vs_oracle(variant, dtype, d_model, reps, sequenced):
    """forward_bidirectional(x, lengths) on the valid frames of every utterance equals the oracle run at that utterance's
    length, for both forward-scan kernels (forced), both dtypes, the eager native block (bf16) and the sequenced
    Functions; d_inner 160 does not fill the 32-channel groups, and 130 utterances of d_inner 288 give the wide kernel
    96-channel CTAs."""
    if dtype == torch.float32 and not sequenced:
        pytest.skip("fp32 always runs the sequenced Functions")
    m, pr = _mamba(d_model, seed=d_model + reps)
    lengths = LENGTHS * reps
    g = torch.Generator().manual_seed(d_model)
    x = torch.randn(len(lengths), max(lengths), d_model, generator=g)
    seq = bm.ops.sequenced_block() if sequenced else bm.ops._NULL
    with bm._lib.tuning(bm._lib.TUNE_SCAN_FWD, variant), torch.no_grad(), _autocast(dtype), seq:
        out = m.forward_bidirectional(x.cuda(), lengths)
    assert out.dtype == dtype
    _check_block(m, pr, x, lengths, out, TOL[dtype])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_backend_varlen_vs_oracle(dtype):
    """Scores of a padded batch with lengths (fp32: the sequenced Functions; bf16 autocast: the native encoder layer and
    the head kernel) against oracle.varlen_oracle.backend_varlen_ref."""
    net, lay, head = _backend()
    lengths = [1, 2, 3, 5, 8, 9, 16, 17, 33, 50, 63, 64]
    g = torch.Generator().manual_seed(4)
    x = torch.randn(len(lengths), 64, 144, generator=g)
    f_ref, s_ref = backend_varlen_ref(lay, head, x.double().cuda(), lengths)
    with torch.no_grad(), _autocast(dtype):
        feats, logits = net(x.cuda(), lengths)
    cmp.check("feats", feats, f_ref, TOL[dtype], cmp.UTT)
    cmp.check("logits", logits, s_ref, TOL[dtype], cmp.UTT)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_graphed_forward_serves_every_length_mix(dtype):
    """One GraphedForward captured with a lengths example and replayed with two other length vectors (a list and a CUDA
    tensor) and new frames: scores match the oracle for each."""
    net, lay, head = _backend()
    T, B = 48, 10

    def score(x, lengths):
        with _autocast(dtype):
            return net(x, lengths)

    g = torch.Generator().manual_seed(5)
    runner = bm.GraphedForward(score, torch.zeros(B, T, 144, device="cuda"), lengths=[T] * B)
    for lengths in ([1, 3, 4, 9, 16, 17, 30, 47, 48, 48], torch.tensor([48, 2, 8, 33, 1, 25, 40, 7, 16, 31], device="cuda")):
        x = torch.randn(B, T, 144, generator=g)
        feats, logits = runner.run(x.cuda(), lengths)
        f_ref, s_ref = backend_varlen_ref(lay, head, x.double().cuda(), [int(v) for v in lengths])
        cmp.check("feats", feats, f_ref, TOL[dtype], cmp.UTT)
        cmp.check("logits", logits, s_ref, TOL[dtype], cmp.UTT)


def _padded(x, lengths, value):
    x = x.clone()
    for b, n in enumerate(lengths):
        x[b, n:] = value
    return x


@pytest.mark.parametrize("path", ["fp32", "bf16_native", "bf16_graphed"])
def test_padding_never_leaks(path):
    """NaN or 1e4 in the padded frames: features and logits are bit-identical to the zero-padded run, and finite."""
    net, _, _ = _backend()
    lengths = [1, 2, 3, 9, 17, 31, 40, 40]
    g = torch.Generator().manual_seed(6)
    x = torch.randn(len(lengths), 40, 144, generator=g)
    dtype = torch.float32 if path == "fp32" else torch.bfloat16
    if path == "bf16_graphed":
        def score(xx, ll):
            with _autocast(dtype):
                return net(xx, ll)
        runner = bm.GraphedForward(score, torch.zeros_like(x, device="cuda"), lengths=lengths)
        run = lambda xx: [t.clone() for t in runner.run(xx, lengths)]
    else:
        def run(xx):
            with torch.no_grad(), _autocast(dtype):
                return net(xx, lengths)
    base = run(_padded(x, lengths, 0.0).cuda())
    assert all(t.isfinite().all() for t in base)
    for value in (float("nan"), 1e4):
        out = run(_padded(x, lengths, value).cuda())
        for a, b in zip(out, base):
            assert torch.equal(a, b), (path, value)


def test_zero_length_utterance_scores_as_zero_features():
    """A device lengths vector is trusted: a zero-length utterance pools to zero features (logits = classifier bias), with
    no NaN, and does not disturb its neighbours."""
    net, _, _ = _backend()
    g = torch.Generator().manual_seed(7)
    x = torch.randn(3, 24, 144, generator=g).cuda()
    with torch.no_grad():
        feats, logits = net(x, torch.tensor([24, 0, 11], device="cuda", dtype=torch.int32))
        f2, l2 = net(x[[0, 2]], [24, 11])
    assert torch.equal(feats[1], torch.zeros_like(feats[1]))
    assert torch.equal(logits[1], net.classifier.bias.detach())
    assert cmp.rel(feats[[0, 2]], f2) < 1e-6 and cmp.rel(logits[[0, 2]], l2) < 1e-6


@pytest.mark.parametrize("path", ["fp32", "bf16_native", "bf16_sequenced"])
def test_full_lengths_equal_the_fixed_length_path_bitwise(path):
    """lengths == T for every utterance gives exactly the bits of lengths=None: block and backend, each path."""
    dtype = torch.float32 if path == "fp32" else torch.bfloat16
    seq = bm.ops.sequenced_block if path == "bf16_sequenced" else (lambda: bm.ops._NULL)
    m, _ = _mamba(144, seed=8)
    net, _, _ = _backend()
    g = torch.Generator().manual_seed(8)
    x = torch.randn(6, 57, 144, generator=g).cuda()
    full = [57] * 6
    with torch.no_grad(), _autocast(dtype), seq():
        assert torch.equal(m.forward_bidirectional(x, full), m.forward_bidirectional(x))
        for a, b in zip(net(x, full), net(x)):
            assert torch.equal(a, b)
    if path == "bf16_sequenced":
        def score(xx, ll=None):
            with _autocast(dtype):
                return net(xx, ll)
        with_len = [t.clone() for t in bm.GraphedForward(score, x, lengths=full).run()]
        without = bm.GraphedForward(score, x).run()
        for a, b in zip(with_len, without):
            assert torch.equal(a, b)


def test_eer_identity_at_mixed_lengths():
    """~2 000 utterances padded to 201 frames with lengths from a small fixed set (the fp64 oracle runs batched per
    length): fp32 scores within 1e-4 and the IDENTICAL EER; bf16 within the bounds of test_eer_identity_full_scoring_set."""
    n_utt, T = 2000, 201
    layers = [orc.init_encoder_params(144, 16, seed=20 + i) for i in range(4)]
    head = orc.init_head_params(144, seed=5)
    g = torch.Generator().manual_seed(2022)
    feats = torch.randn(n_utt, T, 144, generator=g)
    labels = (torch.rand(n_utt, generator=g) < 0.1).numpy()
    choice = torch.tensor([60, 101, 150, 201])
    lengths = choice[torch.randint(0, 4, (n_utt,), generator=g)]
    with torch.no_grad():
        lay_d = [{k: v.double().cuda() for k, v in p.items()} for p in layers]
        head_d = {k: v.double().cuda() for k, v in head.items()}
        s_ref = backend_varlen_ref(lay_d, head_d, feats.double().cuda(), lengths.tolist())[1][:, 1].cpu().numpy()
    net = bm.BiMambaBackend(144, 4, 16).cuda().eval()
    sd = {f"backbone_layers.{i}.{k}": v for i, p in enumerate(layers) for k, v in p.items()}
    sd.update(head)
    net.load_state_dict(sd, strict=True)
    eer_ref, _ = orc.compute_eer_ref(s_ref[labels], s_ref[~labels])
    out = {}
    for name, dtype in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        with torch.no_grad(), _autocast(dtype):
            s = torch.cat([net(feats[i:i + 256].cuda(), lengths[i:i + 256])[1][:, 1].float() for i in range(0, n_utt, 256)])
        s = s.cpu().numpy().astype(np.float64)
        eer, _ = orc.compute_eer_ref(s[labels], s[~labels])
        out[name] = (float(np.abs(s - s_ref).max()), eer)
    print("EER identity set, mixed lengths:", {"ref_eer": eer_ref, **out})
    scale = max(1.0, float(np.abs(s_ref).max()))
    assert out["fp32"][0] < 1e-4 * scale and out["fp32"][1] == eer_ref
    assert out["bf16"][0] < 2e-2 * scale and abs(out["bf16"][1] - eer_ref) < 5e-3


def test_lengths_with_autograd_recording_raise():
    m, _ = _mamba(144, seed=9)
    net, _, _ = _backend()
    x = torch.randn(2, 10, 144, device="cuda")
    with pytest.raises(NotImplementedError):
        m.forward_bidirectional(x, [10, 4])
    with pytest.raises(NotImplementedError):
        net(x, [10, 4])
    with pytest.raises(NotImplementedError), torch.autocast("cuda", dtype=torch.bfloat16):
        net(x, [10, 4])
    with pytest.raises(NotImplementedError):
        bm.backend_head(net, x, [10, 4])
    with pytest.raises(NotImplementedError):
        bm.bimamba_inner_fn(x.requires_grad_(True), *[p.detach() for p in (
            m.in_proj.weight, m.conv1d.weight, m.conv1d.bias, m.x_proj.weight, m.dt_proj.weight, m.dt_proj.bias, m.A_log,
            m.D, m.out_proj.weight)], lengths=[10, 4])
