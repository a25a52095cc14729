"""Mixup on the host side (no GPU): the oracle's contract against a hand-built per-pair loop, the CPU form of mixup_batch
with lengths, the device-record form of mixup_loss, Phase6TrainStep on (x, y, lengths) micro-batches, and the C ABI of
bimamba_mixup_frames (argument errors as codes, a C99 host that compiles with -Wall -Werror)."""
import ctypes as C
import importlib
import os
import subprocess

import pytest
import torch
import torch.nn as nn

import bimamba_b200 as bm
from oracle.mixup_oracle import mixup_ref

tr = importlib.import_module("robust-audio-deepfake-evolution_b200.training")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bimamba.h")
FAKE = 4096          # a non-null device address: every call below must fail before touching it


def _pad(x, lengths, value):
    x = x.clone()
    for b, n in enumerate(lengths):
        x[b, n:] = value
    return x


def test_mixup_ref_against_a_per_pair_loop():
    g = torch.Generator().manual_seed(0)
    B, T, Cc = 6, 9, 3
    lengths = [9, 4, 0, 1, 7, 4]
    perm = [3, 0, 5, 2, 4, 1]
    lam = 0.37
    clean = torch.randn(B, T, Cc, generator=g, dtype=torch.float64)
    for pad in (0.0, 1e4, float("nan")):
        x = _pad(clean, lengths, pad)
        out, m = mixup_ref(x, perm, lam, lengths)
        assert out.dtype == torch.float64 and torch.isfinite(out).all()
        for b in range(B):
            p = perm[b]
            mb = max(lengths[b], lengths[p])
            assert int(m[b]) == mb
            for t in range(T):
                want = torch.zeros(Cc, dtype=torch.float64)
                if t < lengths[b]:
                    want = want + lam * clean[b, t]
                if t < lengths[p]:
                    want = want + (1 - lam) * clean[p, t]
                assert torch.allclose(out[b, t], want, rtol=0, atol=1e-15), (b, t)
            assert bool((out[b, mb:] == 0).all())
    # the identity permutation is the frame mask (lam x + (1 - lam) x over the clip's own frames)
    x = _pad(clean, lengths, float("nan"))
    out, m = mixup_ref(x, list(range(B)), lam, lengths)
    assert m.tolist() == lengths
    assert torch.allclose(out, _pad(clean, lengths, 0.0), rtol=1e-15, atol=0)
    # lengths are clamped to [0, T]
    out2, m2 = mixup_ref(x, perm, lam, [40, 4, -3, 1, 7, 4])
    assert m2.tolist() == mixup_ref(x, perm, lam, [9, 4, 0, 1, 7, 4])[1].tolist()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_torch_expression_form_reduces_to_the_fixed_length_expression(dtype):
    g = torch.Generator().manual_seed(1)
    x = torch.randn(5, 11, 7, generator=g).to(dtype)
    perm = torch.randperm(5, generator=g)
    for lam in (0.0, 1.0, 0.3, 1e-7, 1 - 1e-7):
        out, m = mixup_ref(x, perm, lam, None, exact=False)
        assert torch.equal(out, lam * x + (1.0 - lam) * x[perm]) and m.tolist() == [11] * 5
        full, _ = mixup_ref(x, perm, lam, [11] * 5, exact=False)
        assert torch.equal(full, out)


def test_mixup_batch_with_lengths_on_the_cpu_is_the_contract():
    g = torch.Generator().manual_seed(2)
    lengths = [8, 3, 5, 1]
    x = _pad(torch.randn(4, 8, 2, generator=g), lengths, float("nan"))
    y = torch.tensor([0, 1, 1, 0])
    perm = torch.randperm(4, generator=torch.Generator().manual_seed(3))
    mx, ya, yb, lam, ml = tr.mixup_batch(x, y, 1.0, torch.Generator().manual_seed(3), 0.6, lengths)
    ref, m = mixup_ref(x, perm, 0.6, lengths, exact=False)
    assert torch.equal(mx, ref) and ml.tolist() == m.tolist() and torch.equal(yb, y[perm]) and lam == 0.6
    # an explicit index gives the same; one sample comes back unchanged with its lengths
    again = tr.mixup_batch(x, y, 1.0, None, 0.6, lengths, index=perm)
    assert torch.equal(again[0], mx)
    one = tr.mixup_batch(x[:1], y[:1], 1.0, lengths=[8])
    assert one[3] == 1.0 and one[4] == [8] and torch.equal(one[0], x[:1])
    assert len(tr.mixup_batch(x, y, 1.0, lam=0.5)) == 4


def test_mixup_loss_device_record_gives_the_float_bits():
    g = torch.Generator().manual_seed(4)
    for _ in range(200):
        la, lb = torch.rand(2, generator=g) * 3
        lam = float(torch.rand((), generator=g, dtype=torch.float64))
        rec = torch.tensor([lam, 1.0 - lam], dtype=torch.float32)
        f = lambda out, feats, y: la if y == 0 else lb
        assert torch.equal(tr.mixup_loss(f, None, None, 0, 1, rec), tr.mixup_loss(f, None, None, 0, 1, lam))
    # a 0-d lam weights with 1 - lam
    lam_t = torch.tensor(0.25)
    f = lambda out, feats, y: torch.tensor(2.0) if y == 0 else torch.tensor(6.0)
    assert float(tr.mixup_loss(f, None, None, 0, 1, lam_t)) == 0.25 * 2 + 0.75 * 6


class _Clip(nn.Module):
    """(features, logits) over a right-padded (B, T, 6) batch: masked mean of a projection over each clip's frames."""

    def __init__(self):
        super().__init__()
        torch.manual_seed(0)
        self.feature_projection = nn.Linear(6, 8)
        self.classifier = nn.Linear(8, 2)

    def forward(self, x, lengths=None, *, mask_padding=False):
        B, T = x.shape[:2]
        h = torch.tanh(self.feature_projection(x))
        n = torch.full((B,), T) if lengths is None else torch.as_tensor(lengths)
        if mask_padding:
            h = h.masked_fill((torch.arange(T) >= n.view(-1, 1)).unsqueeze(-1), 0.0)
        f = h.sum(1) / n.view(-1, 1).to(h.dtype)
        return f, self.classifier(f)


def _ce(out, feats, y):
    return nn.functional.cross_entropy(out.float(), y, weight=torch.tensor([0.1, 0.9]))


def _run(batches, lengths):
    m = _Clip()
    opt = torch.optim.AdamW(m.parameters(), lr=1e-2, weight_decay=1e-4)
    step = tr.Phase6TrainStep(m, opt, _ce, autocast_dtype=None, fgm=tr.FGM(m, "feature_projection", 0.5),
                              mixup_alpha=1.0, accumulation_steps=2)
    mbs = [(x, y) if lengths is None else (x, y, n) for (x, y), n in zip(batches, lengths or [None] * len(batches))]
    torch.manual_seed(11)
    loss = step(mbs, generator=torch.Generator().manual_seed(9))
    return loss, [p.detach().clone() for p in m.parameters()]


def test_phase6_step_with_lengths_reduces_to_the_fixed_length_step():
    gen = torch.Generator().manual_seed(5)
    batches = [(torch.randn(4, 7, 6, generator=gen), torch.randint(0, 2, (4,), generator=gen)) for _ in range(2)]
    loss_a, pa = _run(batches, None)
    loss_b, pb = _run(batches, [[7] * 4, [7] * 4])
    assert torch.equal(loss_a, loss_b)
    for p, q in zip(pa, pb):
        assert torch.equal(p, q)


def test_phase6_step_with_lengths_equals_the_loop_body():
    """Mixup on each clip's frames, the model on the mixed lengths with mask_padding=True in both passes of FGM."""
    gen = torch.Generator().manual_seed(6)
    lengths = [[7, 2, 5, 3], [1, 7, 7, 4]]
    batches = [(_pad(torch.randn(4, 7, 6, generator=gen), n, float("nan")), torch.randint(0, 2, (4,), generator=gen))
               for n in lengths]
    loss, got = _run(batches, lengths)
    assert torch.isfinite(loss)
    b = _Clip()
    opt = torch.optim.AdamW(b.parameters(), lr=1e-2, weight_decay=1e-4)
    torch.manual_seed(11)
    g2 = torch.Generator().manual_seed(9)
    total = None
    for (x, y), n in zip(batches, lengths):
        lam = float(torch.distributions.Beta(1.0, 1.0).sample())
        idx = torch.randperm(4, generator=g2)
        mx, ml = mixup_ref(x, idx, lam, n, exact=False)
        ya, yb = y, y[idx]

        def loss_fn():
            out = b(mx, ml, mask_padding=True)[1]
            return (lam * _ce(out, None, ya) + (1.0 - lam) * _ce(out, None, yb)) / 2
        l0 = loss_fn()
        l0.backward()
        total = l0.detach() if total is None else total + l0.detach()
        w, bias = b.feature_projection.weight, b.feature_projection.bias
        keep = (w.data.clone(), bias.data.clone())
        w.data.add_(0.5 * w.grad / w.grad.norm())
        bias.data.add_(0.5 * bias.grad / bias.grad.norm())
        loss_fn().backward()
        w.data, bias.data = keep
    torch.nn.utils.clip_grad_norm_(b.parameters(), 3.0)
    opt.step()
    assert torch.allclose(loss, total, rtol=1e-6)
    for p, q in zip(got, b.parameters()):
        assert torch.allclose(p, q, atol=1e-6)


def test_mixup_frames_is_declared_exported_and_typed():
    assert "bimamba_mixup_frames" in bm._lib.EXPORTS
    with open(HEADER) as f:
        assert "int bimamba_mixup_frames(" in f.read()
    lib = bm._lib.load()
    assert lib.bimamba_mixup_frames.restype is C.c_int and len(lib.bimamba_mixup_frames.argtypes) == 11


def test_mixup_frames_argument_errors_are_codes():
    lib = bm._lib.load()
    f = lib.bimamba_mixup_frames
    assert f(FAKE, FAKE, None, FAKE, None, None, 2, 5, 144, 0, None) == -1           # no perm
    assert f(FAKE, FAKE, FAKE, None, None, None, 2, 5, 144, 0, None) == -1           # no mix
    assert f(None, FAKE, FAKE, FAKE, None, None, 2, 5, 144, 0, None) == -1           # no x
    assert f(FAKE, None, FAKE, FAKE, None, None, 2, 5, 144, 0, None) == -1           # no out
    assert f(FAKE, FAKE, FAKE, FAKE, FAKE, None, 2, 5, 144, 0, None) == -1           # lengths in, nowhere to write them
    assert f(FAKE, FAKE, FAKE, FAKE, None, None, -1, 5, 144, 0, None) == -3
    assert f(FAKE, FAKE, FAKE, FAKE, None, None, 2, -5, 144, 0, None) == -3
    assert f(FAKE, FAKE, FAKE, FAKE, None, None, 2, 5, -1, 0, None) == -3
    assert f(FAKE, FAKE, FAKE, FAKE, None, None, 2, 5, 144, 3, None) == -3           # bad dtype
    assert f(None, None, None, None, None, None, 0, 5, 144, 0, None) == 0            # empty batch


def test_c_host_calling_mixup_frames_compiles_and_links(tmp_path):
    prog = tmp_path / "host_mixup.c"
    prog.write_text(f"""#include <stdio.h>
#include "{HEADER}"
/* Mixup of a padded batch of waveforms before the training step: perm and {{lam, 1 - lam}} already on the device */
int mix_batch(void* stream, const float* wav, float* mixed, const int32_t* perm, const float* mix,
              const int32_t* seqlens, int32_t* mixed_seqlens) {{
  int rc = bimamba_mixup_frames(wav, mixed, perm, mix, seqlens, mixed_seqlens, 64, 64600, 1, BIMAMBA_F32, stream);
  if (rc) fprintf(stderr, "%s\\n", bimamba_last_error());
  return rc;
}}
int main(void) {{
  printf("%d %d\\n", bimamba_abi_version(), mix_batch(0, 0, 0, 0, 0, 0, 0));
  return 0;
}}
""")
    exe = tmp_path / "host_mixup"
    lib = bm._lib.LIB_PATH
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", str(prog), "-o", str(exe), lib,
                           "-Wl,-rpath," + os.path.dirname(lib)])
    out = subprocess.check_output([str(exe)], text=True).split()
    assert int(out[0]) == bm._lib.ABI_VERSION == 12 and int(out[1]) == -1
