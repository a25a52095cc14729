"""Host-side checks of variable-length scoring (no device needed): argument errors of the _varlen entry points come back as
codes, a C99 host calling them compiles with -Wall -Werror and links, and host-side lengths are validated in Python."""
import ctypes as C
import os
import subprocess

import pytest
import torch

import bimamba_b200 as bm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bimamba.h")
FAKE = 4096          # a non-null device address: every call below must fail before touching it


def test_varlen_argument_errors_are_codes():
    lib = bm._lib.load()
    # block / layer: forward-only, whatever else the descriptor holds
    d = bm._lib.BlockDesc()
    d.batch, d.seqlen, d.d_model, d.d_inner, d.dt_rank, d.d_conv, d.ndir = 2, 5, 144, 288, 9, 4, 2
    d.io_dtype, d.save_for_backward = bm._lib.BF16, 1
    assert lib.bimamba_block_fwd_varlen(C.byref(d), FAKE, None) == -9
    assert b"forward-only" in lib.bimamba_last_error()
    assert lib.bimamba_block_fwd_varlen(C.byref(d), None, None) == -7       # NULL seqlens = the fixed-length call
    d.save_for_backward = 0
    assert lib.bimamba_block_fwd_varlen(C.byref(d), FAKE, None) == -7       # null operands
    assert lib.bimamba_block_fwd_varlen(None, FAKE, None) == -1
    ld = bm._lib.LayerDesc()
    k = ld.block
    k.batch, k.seqlen, k.d_model, k.d_inner, k.dt_rank, k.d_conv, k.ndir, k.io_dtype = 2, 5, 144, 288, 9, 4, 2, bm._lib.BF16
    k.save_for_backward = 1
    ld.d_ff, ld.x_dtype = 576, bm._lib.F32
    assert lib.bimamba_layer_fwd_varlen(C.byref(ld), FAKE, None) == -9
    assert b"forward-only" in lib.bimamba_last_error()
    k.save_for_backward = 0
    assert lib.bimamba_layer_fwd_varlen(C.byref(ld), FAKE, None) == -7     # null operands
    assert lib.bimamba_layer_fwd_varlen(None, FAKE, None) == -1
    # scan: no checkpoints with lengths (validated before any launch)
    s = bm._lib.ScanDesc()
    s.batch, s.ndir, s.dim, s.seqlen, s.dstate, s.group_channels = 2, 2, 32, 40, 16, 32
    s.u = s.A = s.bc = s.delta = s.out = s.ckpt = FAKE
    assert lib.bimamba_selective_scan_fwd_varlen(C.byref(s), FAKE, None) == -9
    assert b"checkpoints" in lib.bimamba_last_error()
    assert lib.bimamba_selective_scan_fwd_varlen(None, FAKE, None) == -1
    s.batch = 0
    assert lib.bimamba_selective_scan_fwd_varlen(C.byref(s), FAKE, None) == 0
    # conv / head
    assert lib.bimamba_causal_conv1d_fwd_varlen(None, None, None, None, FAKE, 2, 2, 8, 5, 4, 0, 0, 0, 0, 0, 0, 1, None) == -1
    assert lib.bimamba_causal_conv1d_fwd_varlen(None, None, None, None, FAKE, 0, 2, 8, 5, 4, 0, 0, 0, 0, 0, 0, 1, None) == 0
    assert lib.bimamba_head_fwd_varlen(None, None, None, None, None, None, None, None, None, FAKE, 2, 5, 144, 2, 1e-5, 0,
                                       None) == -1
    assert lib.bimamba_head_fwd_varlen(None, None, None, None, None, None, None, None, None, FAKE, 0, 5, 144, 2, 1e-5, 0,
                                       None) == 0


def test_c_host_calling_the_varlen_entries_compiles_and_links(tmp_path):
    prog = tmp_path / "host_varlen.c"
    prog.write_text(f"""#include <stdio.h>
#include "{HEADER}"
int score(void* stream, const float* x, float* out, const int32_t* seqlens) {{
  bimamba_layer_desc l = {{0}};
  l.x = x; l.out = out; l.eps1 = l.eps2 = 1e-5f; l.d_ff = 576; l.x_dtype = BIMAMBA_F32;
  l.block.batch = 256; l.block.seqlen = 499; l.block.d_model = 144; l.block.d_inner = 288; l.block.dt_rank = 9;
  l.block.d_conv = 4; l.block.ndir = 2; l.block.io_dtype = BIMAMBA_BF16; l.block.save_for_backward = 0;
  l.workspace_bytes = bimamba_layer_fwd_workspace_bytes(256, 499, 144, 288, 576, 2, BIMAMBA_BF16, 0);
  int rc = bimamba_layer_fwd_varlen(&l, seqlens, stream);
  if (rc) fprintf(stderr, "%s\\n", bimamba_last_error());
  return rc;
}}
int others(void* stream, const int32_t* seqlens) {{
  bimamba_block_desc b = {{0}};
  bimamba_scan_desc s = {{0}};
  float feats[2], logits[2];
  int rc = bimamba_block_fwd_varlen(&b, seqlens, stream);
  rc = rc ? rc : bimamba_selective_scan_fwd_varlen(&s, seqlens, stream);
  rc = rc ? rc : bimamba_causal_conv1d_fwd_varlen(0, 0, 0, 0, seqlens, 1, 2, 8, 5, 4, 0, 0, 0, 0, 0, BIMAMBA_BF16,
                                                  BIMAMBA_FLAG_SILU, stream);
  return rc ? rc : bimamba_head_fwd_varlen(0, 0, 0, 0, 0, 0, 0, feats, logits, seqlens, 1, 5, 144, 2, 1e-5f,
                                           BIMAMBA_F32, stream);
}}
int main(void) {{
  printf("%d %d %d\\n", bimamba_abi_version(), score(0, 0, 0, 0), others(0, 0));
  return 0;
}}
""")
    exe = tmp_path / "host_varlen"
    lib = bm._lib.LIB_PATH
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", str(prog), "-o", str(exe), lib,
                           "-Wl,-rpath," + os.path.dirname(lib)])
    # argument validation only (null operands -> error code before any CUDA call): safe without a GPU
    out = subprocess.check_output([str(exe)], text=True).split()
    assert int(out[0]) == bm._lib.ABI_VERSION == 12 and int(out[1]) < 0 and int(out[2]) < 0


@pytest.mark.parametrize("lengths,msg", [([0, 3], "1..5"), ([1, 6], "1..5"), ([2], "integer frame counts"),
                                         ([[1, 2]], "integer frame counts"), ([1.0, 2.0], "integer frame counts"),
                                         (torch.tensor([3, 9]), "1..5")])
def test_host_side_lengths_are_validated(lengths, msg):
    with pytest.raises(ValueError, match=msg):
        bm.ops.seqlens_tensor(lengths, 2, 5, "cpu")
    x = torch.randn(2, 5, 144)
    # the public entry points validate before they look for a device
    with pytest.raises(ValueError, match=msg):
        bm.Mamba(144, 16).forward_bidirectional(x, lengths)
    with pytest.raises(ValueError, match=msg):
        bm.PN_BiMambas_Encoder(144, 16)(x, lengths)
    net = bm.BiMambaBackend(144, 1, 16).eval()
    with pytest.raises(ValueError, match=msg):
        net(x, lengths)
    with pytest.raises(ValueError, match=msg):
        bm.backend_head(net, x, lengths)


def test_valid_host_lengths_become_an_int32_vector():
    for lengths in ([5, 1], (5, 1), torch.tensor([5, 1]), torch.tensor([5, 1], dtype=torch.int16)):
        t = bm.ops.seqlens_tensor(lengths, 2, 5, "cpu")
        assert t.dtype == torch.int32 and t.tolist() == [5, 1]
    assert bm.ops.seqlens_tensor(None, 2, 5, "cpu") is None
    with pytest.raises(RuntimeError, match="no CPU fallback"):       # valid lengths, then the usual refusal
        bm.Mamba(144, 16).forward_bidirectional(torch.randn(2, 5, 144), [5, 1])
