"""Host-side checks of variable-length training (no device needed): argument errors of the new entry points come back as
codes, a C99 host calling every one of them compiles with -Wall -Werror and links, mask_padding is validated before any
device lookup, and the gradient oracle's per-length batching equals a per-utterance loop."""
import ctypes as C
import os
import subprocess

import pytest
import torch
import torch.nn.functional as F

import bimamba_b200 as bm
from oracle import bimamba_oracle as orc
from oracle.varlen_train_oracle import backend_logits_fn, varlen_loss_and_grads_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bimamba.h")
FAKE = 4096          # a non-null device address: every call below must fail before touching it


def test_training_entry_argument_errors_are_codes():
    lib = bm._lib.load()
    s = bm._lib.ScanDesc()
    s.batch, s.ndir, s.dim, s.seqlen, s.dstate, s.group_channels = 2, 2, 32, 40, 16, 32
    assert lib.bimamba_selective_scan_fwd_varlen_train(None, FAKE, None) == -1
    assert lib.bimamba_selective_scan_fwd_varlen_train(C.byref(s), FAKE, None) == -7        # null operands
    assert lib.bimamba_selective_scan_bwd_varlen(None, FAKE, None) == -1
    s.u = s.A = s.bc = s.delta = s.out = FAKE
    assert lib.bimamba_selective_scan_bwd_varlen(C.byref(s), FAKE, None) == -8               # no backward operands
    s.dout = s.du = s.ddelta = s.dbc_part = s.dA_part = FAKE
    assert lib.bimamba_selective_scan_bwd_varlen(C.byref(s), FAKE, None) == -9               # no checkpoints
    s.batch = 0
    assert lib.bimamba_selective_scan_bwd_varlen(C.byref(s), FAKE, None) == 0
    assert lib.bimamba_causal_conv1d_bwd_varlen(None, None, None, None, None, None, None, None, FAKE, 2, 2, 8, 5, 4,
                                                0, 0, 0, 0, 0, 0, 0, 0, 1, None) == -1
    assert lib.bimamba_causal_conv1d_bwd_varlen(FAKE, FAKE, None, FAKE, FAKE, FAKE, None, FAKE, FAKE, 2, 2, 8, 5, 4,
                                                0, 0, 0, 0, 0, 0, 0, 0, 1, None) == -1               # dz_in without dz_out
    assert lib.bimamba_head_pool_bwd_varlen(None, None, None, None, None, None, None, None, FAKE, 2, 5, 144, 1e-5, 0,
                                            None) == -1
    assert lib.bimamba_head_pool_bwd_varlen(FAKE, FAKE, FAKE, FAKE, None, FAKE, FAKE, FAKE, FAKE, 2, 5, 300, 1e-5, 0,
                                            None) == -3
    assert lib.bimamba_mask_frames(None, FAKE, FAKE, 2, 5, 144, 0, None) == -1
    assert lib.bimamba_mask_frames(FAKE, FAKE, None, 2, 5, 144, 0, None) == -1
    assert lib.bimamba_mask_frames(FAKE, FAKE, FAKE, 2, 5, 144, 7, None) == -3
    assert lib.bimamba_mask_frames(None, None, None, 0, 5, 144, 0, None) == 0
    # block / layer: the training forms accept save_for_backward and check the descriptor as the fixed-length calls do
    d = bm._lib.BlockDesc()
    d.batch, d.seqlen, d.d_model, d.d_inner, d.dt_rank, d.d_conv, d.ndir = 2, 5, 144, 288, 9, 4, 2
    d.io_dtype, d.save_for_backward = bm._lib.BF16, 1
    assert lib.bimamba_block_fwd_varlen_train(C.byref(d), FAKE, None) == -7                   # null operands
    assert lib.bimamba_block_fwd_varlen_train(None, FAKE, None) == -1
    g = bm._lib.BlockGrads()
    assert lib.bimamba_block_bwd_varlen(None, C.byref(g), FAKE, None) == -1
    ld = bm._lib.LayerDesc()
    k = ld.block
    k.batch, k.seqlen, k.d_model, k.d_inner, k.dt_rank, k.d_conv, k.ndir, k.io_dtype = 2, 5, 144, 288, 9, 4, 2, bm._lib.BF16
    k.save_for_backward = 1
    ld.d_ff, ld.x_dtype = 576, bm._lib.F32
    assert lib.bimamba_layer_fwd_varlen_train(C.byref(ld), FAKE, None) == -7
    assert lib.bimamba_layer_bwd_varlen(None, None, FAKE, None) == -1


def test_c_host_calling_the_training_entries_compiles_and_links(tmp_path):
    prog = tmp_path / "host_varlen_train.c"
    prog.write_text(f"""#include <stdio.h>
#include "{HEADER}"
/* one masked training step of an encoder layer, as bimamba.h describes it */
int train_layer(void* stream, float* x, float* out, float* dout, const int32_t* seqlens) {{
  bimamba_layer_desc l = {{0}};
  bimamba_layer_grads g = {{0}};
  l.x = x; l.out = out; l.eps1 = l.eps2 = 1e-5f; l.d_ff = 576; l.x_dtype = BIMAMBA_F32;
  l.block.batch = 64; l.block.seqlen = 201; l.block.d_model = 144; l.block.d_inner = 288; l.block.dt_rank = 9;
  l.block.d_conv = 4; l.block.ndir = 2; l.block.io_dtype = BIMAMBA_BF16; l.block.save_for_backward = 1;
  l.workspace_bytes = bimamba_layer_fwd_workspace_bytes(64, 201, 144, 288, 576, 2, BIMAMBA_BF16, 1);
  g.dout = dout;
  int rc = bimamba_mask_frames(x, x, seqlens, 64, 201, 144, BIMAMBA_F32, stream);
  rc = rc ? rc : bimamba_layer_fwd_varlen_train(&l, seqlens, stream);
  rc = rc ? rc : bimamba_mask_frames(out, out, seqlens, 64, 201, 144, BIMAMBA_F32, stream);
  rc = rc ? rc : bimamba_mask_frames(dout, dout, seqlens, 64, 201, 144, BIMAMBA_F32, stream);
  rc = rc ? rc : bimamba_layer_bwd_varlen(&l, &g, seqlens, stream);
  if (rc) fprintf(stderr, "%s\\n", bimamba_last_error());
  return rc;
}}
int others(void* stream, const int32_t* seqlens) {{
  bimamba_block_desc b = {{0}};
  bimamba_block_grads bg = {{0}};
  bimamba_scan_desc s = {{0}};
  float feats[2];
  int rc = bimamba_block_fwd_varlen_train(&b, seqlens, stream);
  rc = rc ? rc : bimamba_block_bwd_varlen(&b, &bg, seqlens, stream);
  rc = rc ? rc : bimamba_selective_scan_fwd_varlen_train(&s, seqlens, stream);
  rc = rc ? rc : bimamba_selective_scan_bwd_varlen(&s, seqlens, stream);
  rc = rc ? rc : bimamba_causal_conv1d_bwd_varlen(0, 0, 0, 0, 0, 0, 0, 0, seqlens, 1, 2, 8, 5, 4, 0, 0, 0, 0, 0, 0, 0,
                                                  BIMAMBA_BF16, BIMAMBA_FLAG_SILU, stream);
  return rc ? rc : bimamba_head_pool_bwd_varlen(0, 0, 0, 0, 0, feats, 0, 0, seqlens, 1, 5, 144, 1e-5f, BIMAMBA_F32,
                                                stream);
}}
int main(void) {{
  printf("%d %d %d\\n", bimamba_abi_version(), train_layer(0, 0, 0, 0, 0), others(0, 0));
  return 0;
}}
""")
    exe = tmp_path / "host_varlen_train"
    lib = bm._lib.LIB_PATH
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", str(prog), "-o", str(exe), lib,
                           "-Wl,-rpath," + os.path.dirname(lib)])
    # argument validation only (null operands -> error code before any CUDA call): safe without a GPU
    out = subprocess.check_output([str(exe)], text=True).split()
    assert int(out[0]) == bm._lib.ABI_VERSION == 12 and int(out[1]) < 0 and int(out[2]) < 0


def test_mask_padding_needs_lengths_and_lengths_are_validated_first():
    x = torch.randn(2, 5, 144)
    net = bm.BiMambaBackend(144, 1, 16)
    calls = [lambda lens, **kw: bm.Mamba(144, 16).forward_bidirectional(x, lens, **kw),
             lambda lens, **kw: bm.PN_BiMambas_Encoder(144, 16)(x, lens, **kw),
             lambda lens, **kw: net(x, lens, **kw),
             lambda lens, **kw: net.forward_features(x, lens, **kw),
             lambda lens, **kw: bm.backend_head(net, x, lens, **kw)]
    for call in calls:
        with pytest.raises(ValueError, match="mask_padding=True needs lengths"):
            call(None, mask_padding=True)
        with pytest.raises(ValueError, match="1..5"):
            call([0, 3], mask_padding=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):       # valid lengths, then the usual refusal
        bm.Mamba(144, 16).forward_bidirectional(x, [5, 1], mask_padding=True)


def test_varlen_gradient_oracle_equals_a_per_utterance_loop():
    layers = [orc.init_encoder_params(16, 4, seed=3, dtype=torch.float64)]
    head = orc.init_head_params(16, seed=3, dtype=torch.float64)
    p = {f"backbone_layers.0.{k}": v for k, v in layers[0].items()}
    p.update(head)
    lengths = [3, 7, 3, 1, 7]
    g = torch.Generator().manual_seed(4)
    x = torch.randn(5, 7, 16, generator=g, dtype=torch.float64)
    x[0, 3:] = float("nan")                                        # padding is never read
    labels = torch.tensor([0, 1, 1, 0, 1])
    ce = lambda lg, idx, n: F.cross_entropy(lg, labels[idx], reduction="sum")
    loss, grads, dx = varlen_loss_and_grads_ref(backend_logits_fn(1), p, x, lengths, ce)
    assert torch.isfinite(dx).all() and bool((dx[0, 3:] == 0).all())
    loss_l, grads_l = 0.0, {k: torch.zeros_like(v) for k, v in p.items()}
    for b, n in enumerate(lengths):
        lb, gb, dxb = varlen_loss_and_grads_ref(backend_logits_fn(1), p, x[b:b + 1], [n],
                                                lambda lg, idx, n_: F.cross_entropy(lg, labels[b:b + 1], reduction="sum"))
        loss_l += float(lb)
        for k in grads_l:
            grads_l[k] += gb[k]
        assert torch.allclose(dx[b], dxb[0], rtol=1e-12, atol=1e-14)
    assert abs(float(loss) - loss_l) <= 1e-12 * abs(loss_l)
    for k in grads:
        assert torch.allclose(grads[k], grads_l[k], rtol=1e-10, atol=1e-13), k
