"""CPU-side checks of the two-stream entry points (bimamba_block_bwd_side, bimamba_layer_fwd_side, bimamba_layer_bwd_side):
the ctypes mirrors of their structs have the C layout, the layer backward's workspace holds one LayerNorm partial buffer
per norm, argument errors are codes, and a C99 host using them compiles and links (nothing runs on a device)."""
import ctypes as C
import os
import subprocess

import pytest

import bimamba_b200 as bm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bimamba.h")


@pytest.mark.parametrize("cname,mirror", [("bimamba_side_stream", "SideStream"), ("bimamba_block_pack", "BlockPack")])
def test_side_stream_struct_layouts_match_header(tmp_path, cname, mirror):
    cls = getattr(bm._lib, mirror)
    fields = [f[0] for f in cls._fields_]
    body = "\n".join(f'  printf("{f} %zu\\n", offsetof({cname}, {f}));' for f in fields)
    prog = tmp_path / "layout.c"
    prog.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "{HEADER}"\nint main(void) {{\n'
                    f'  printf("sizeof %zu\\n", sizeof({cname}));\n{body}\n  return 0;\n}}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", str(prog), "-o", str(exe)])
    out = dict(ln.split() for ln in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(out["sizeof"]) == C.sizeof(cls)
    for f in fields:
        assert int(out[f]) == getattr(cls, f).offset, f


def test_layer_bwd_workspace_has_one_layernorm_partial_buffer_per_norm():
    """norm1's backward (main stream) may run while norm2's dgamma / dbeta sum (side stream) still reads its partials."""
    lib = bm._lib.load()
    up = lambda v: (v + 255) // 256 * 256
    for B, L, dm, D, dff, K, ndir in ((64, 201, 144, 288, 576, 4, 2), (3, 5, 16, 32, 64, 3, 1)):
        M, es = B * L, 2
        tn = max(lib.bimamba_gemm_tn_splits(M, dm, dff), lib.bimamba_gemm_tn_splits(M, dff, dm)) * dm * dff * 4
        own = (4 * up(M * dm * es) + 2 * up(M * dff * es) + up(lib.bimamba_colsum_slices(M) * dff * 4)
               + 2 * up(lib.bimamba_layernorm_bwd_blocks(M) * 2 * dm * 4) + up(tn))
        assert lib.bimamba_layer_bwd_workspace_bytes(B, L, dm, D, dff, K, ndir, bm._lib.BF16) == (
            own + lib.bimamba_block_bwd_workspace_bytes(B, L, dm, D, K, ndir, bm._lib.BF16))


def test_side_stream_argument_errors_are_codes():
    lib = bm._lib.load()
    d = bm._lib.LayerDesc()
    g = bm._lib.LayerGrads()
    s = bm._lib.SideStream()
    # no side stream: the single-stream call's own checks
    assert lib.bimamba_layer_fwd_side(None, None, None, None, None) == -1
    assert lib.bimamba_layer_bwd_side(None, None, None, None, None) == -1
    assert lib.bimamba_block_bwd_side(None, None, None, None, None) == -1
    s.stream = 0x10
    # a side stream without its events, or equal to the main stream, is refused before anything is enqueued
    assert lib.bimamba_layer_bwd_side(C.byref(d), C.byref(g), None, C.byref(s), None) == -11
    assert b"three events" in lib.bimamba_last_error()
    assert lib.bimamba_block_bwd_side(None, None, None, C.byref(s), 0x10) == -11
    assert b"differ" in lib.bimamba_last_error()
    # descriptor errors come before the fork in the forward
    assert lib.bimamba_layer_fwd_side(C.byref(d), None, None, C.byref(s), None) == -3
    k = d.block
    k.batch, k.seqlen, k.d_model, k.d_inner, k.dt_rank, k.d_conv, k.ndir, k.io_dtype = 2, 5, 144, 288, 9, 4, 2, bm._lib.BF16
    d.d_ff, d.x_dtype = 576, bm._lib.F32
    for name in ("x", "out", "norm1_w", "norm1_b", "norm2_w", "norm2_b", "ff_w1", "ff_b1", "ff_w2", "ff_b2", "workspace"):
        setattr(d, name, 256)
    d.workspace_bytes = 1 << 40
    pk = bm._lib.BlockPack()
    assert lib.bimamba_layer_fwd_side(C.byref(d), C.byref(pk), None, None, None) == -7
    assert b"weight pack" in lib.bimamba_last_error()


def test_c99_host_using_the_side_stream_calls_compiles(tmp_path):
    prog = tmp_path / "host.c"
    prog.write_text(f"""#include <stdio.h>
#include "{HEADER}"
int train_layer(void* stream, void* side, void* const ev[3], const float* x, float* out) {{
  bimamba_side_stream s = {{0}};
  s.stream = side; s.events[0] = ev[0]; s.events[1] = ev[1]; s.events[2] = ev[2];
  bimamba_layer_desc l = {{0}};
  l.x = x; l.out = out; l.eps1 = l.eps2 = 1e-5f; l.d_ff = 576; l.x_dtype = BIMAMBA_F32;
  l.block.batch = 8; l.block.seqlen = 201; l.block.d_model = 144; l.block.d_inner = 288; l.block.dt_rank = 9;
  l.block.d_conv = 4; l.block.ndir = 2; l.block.io_dtype = BIMAMBA_BF16; l.block.save_for_backward = 1;
  l.workspace_bytes = bimamba_layer_fwd_workspace_bytes(8, 201, 144, 288, 576, 2, BIMAMBA_BF16, 1);
  bimamba_block_pack p = {{0}};
  bimamba_layer_grads g = {{0}};
  g.workspace_bytes = bimamba_layer_bwd_workspace_bytes(8, 201, 144, 288, 576, 4, 2, BIMAMBA_BF16);
  int rc = bimamba_layer_fwd_side(&l, &p, NULL, &s, stream);
  return rc ? rc : bimamba_layer_bwd_side(&l, &g, NULL, &s, stream);
}}
int block_bwd(void* stream) {{
  bimamba_block_desc d = {{0}};
  bimamba_block_grads g = {{0}};
  return bimamba_block_bwd_side(&d, &g, NULL, NULL, stream);
}}
int main(void) {{
  void* ev[3] = {{0, 0, 0}};
  printf("%d %d %d\\n", bimamba_abi_version(), train_layer(0, 0, ev, 0, 0), block_bwd(0));
  return 0;
}}
""")
    exe = tmp_path / "host"
    lib = bm._lib.LIB_PATH
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", str(prog), "-o", str(exe), lib,
                           "-Wl,-rpath," + os.path.dirname(lib)])
    out = subprocess.check_output([str(exe)], text=True).split()
    assert int(out[0]) == bm._lib.ABI_VERSION and int(out[1]) < 0 and int(out[2]) < 0
