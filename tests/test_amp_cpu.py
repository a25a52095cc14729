"""Host-side checks of the fp16 optimizer step (no GPU): the `struct bimamba_amp` / `struct bimamba_ema_tensor` layouts
against the header, argument errors of the three new entry points come back as codes before any CUDA call, a C99 host
that uses them compiles and links, and DeviceGradScaler takes and refuses constructor arguments as torch.amp.GradScaler
does."""
import ctypes as C
import os
import subprocess

import pytest
import torch

import bimamba_b200 as bm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bimamba.h")
FAKE = 4096          # a non-null pointer the validation must not dereference


def _layout(tmp_path, decl, fields):
    prog = tmp_path / "amp_layout.c"
    body = "\n".join(f'  printf("{f} %zu\\n", offsetof({decl}, {f}));' for f in fields)
    prog.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "{HEADER}"\nint main(void) {{\n'
                    f'  printf("sizeof %zu\\n", sizeof({decl}));\n{body}\n  return 0;\n}}\n')
    exe = tmp_path / "amp_layout"
    subprocess.check_call(["gcc", "-std=c99", str(prog), "-o", str(exe)])
    return {k: int(v) for k, v in (ln.split() for ln in subprocess.check_output([str(exe)], text=True).splitlines())}


def test_amp_record_layout_matches_header(tmp_path):
    cls = bm._lib.AmpRecord
    fields = [f[0] for f in cls._fields_]
    out = _layout(tmp_path, "bimamba_amp", fields)
    assert out["sizeof"] == C.sizeof(cls) == 32
    for f in fields:
        assert out[f] == getattr(cls, f).offset, f
    # the Python side addresses the record as 8 int32 words (amp.py)
    from importlib import import_module
    amp = import_module("robust-audio-deepfake-evolution_b200.amp")
    assert [amp._SCALE, amp._TRACKER, amp._FOUND_INF, amp._TOTAL_NORM, amp._CLIP_COEF] == \
        [getattr(cls, f).offset // 4 for f in fields[:5]]
    assert amp._WORDS * 4 == C.sizeof(cls)
    ema = _layout(tmp_path, "struct bimamba_ema_tensor", ["avg", "n"])
    assert ema == {"sizeof": 16, "avg": 0, "n": 8}       # FusedAdamW writes it as two int64 per entry


def test_new_entry_points_refuse_null_operands_before_any_cuda_call():
    lib = bm._lib.load()
    # statistics: the record is always required; table, block map and partials when there are blocks
    assert lib.bimamba_amp_grad_stats(None, None, 4, 3.0, None, None, None) == -1
    assert lib.bimamba_amp_grad_stats(FAKE, FAKE, 4, 3.0, FAKE, None, None) == -1
    assert lib.bimamba_amp_grad_stats(None, FAKE, 4, 3.0, FAKE, FAKE, None) == -1
    assert lib.bimamba_amp_grad_stats(FAKE, FAKE, 4, 3.0, None, FAKE, None) == -1
    assert lib.bimamba_amp_grad_stats(FAKE, FAKE, -1, 3.0, FAKE, FAKE, None) == -1
    assert lib.bimamba_amp_grad_stats(None, None, 0, 3.0, None, None, None) == -1
    assert b"amp_grad_stats" in lib.bimamba_last_error()
    # the AdamW-with-amp step
    step = lib.bimamba_adamw_amp_step
    assert step(None, None, 0, None, None, None, None, None, 0.0, None) == 0              # empty: no-op success
    assert step(None, FAKE, 4, FAKE, FAKE, FAKE, None, None, 0.0, None) == -1             # no table
    assert step(FAKE, None, 4, FAKE, FAKE, FAKE, None, None, 0.0, None) == -1             # no block map
    assert step(FAKE, FAKE, 4, FAKE, FAKE, None, None, None, 0.0, None) == -1             # hyper / state without amp
    assert step(FAKE, FAKE, 4, None, FAKE, FAKE, None, None, 0.0, None) == -1
    assert step(FAKE, FAKE, 4, FAKE, FAKE, FAKE, FAKE, None, 1e-3, None) == -1            # ema without n_averaged
    assert step(FAKE, FAKE, 4, FAKE, FAKE, FAKE, None, FAKE, 1e-3, None) == -1
    assert step(FAKE, FAKE, 4, None, None, None, None, None, 1e-3, None) == -1            # nothing to do
    assert step(FAKE, FAKE, 4, None, None, None, FAKE, FAKE, 1.5, None) == -2             # weight outside [0, 1]
    assert step(FAKE, FAKE, 4, None, None, None, FAKE, FAKE, float("nan"), None) == -2
    assert b"adamw_amp_step" in lib.bimamba_last_error()
    # the tail
    assert lib.bimamba_amp_update(None, 2.0, 0.5, 2000, None, None) == -1
    assert b"amp_update" in lib.bimamba_last_error()


def test_c99_host_using_the_amp_step_compiles_and_links(tmp_path):
    """A C host running the documented launch order (INTEGRATION.md) compiles with -Wall -Werror and links; with null
    operands every call returns its error code before touching a device."""
    prog = tmp_path / "amp_host.c"
    prog.write_text(f"""#include <stdio.h>
#include "{HEADER}"
/* one optimizer step of the fp16 recipe over ngroups AdamW tables (each group: its slice of the table of all groups) */
int amp_step(const struct bimamba_adamw_tensor* all, const int32_t* all_map, int all_blocks, double* partials,
             const struct bimamba_adamw_tensor* const* tables, const int32_t* const* maps, const int* nblocks,
             const float* const* hyper, float* const* state, const struct bimamba_ema_tensor* const* ema, int ngroups,
             bimamba_amp* amp, int64_t* n_averaged, void* stream) {{
  int rc = bimamba_amp_grad_stats(all, all_map, all_blocks, 3.0f, partials, amp, stream);
  for (int i = 0; rc == 0 && i < ngroups; ++i)
    rc = bimamba_adamw_amp_step(tables[i], maps[i], nblocks[i], hyper[i], state[i], amp, ema ? ema[i] : NULL,
                                n_averaged, 1.0f - 0.999f, stream);
  if (rc == 0) rc = bimamba_amp_update(amp, 2.0, 0.5, 2000, n_averaged, stream);
  if (rc) fprintf(stderr, "%s\\n", bimamba_last_error());
  return rc;
}}
int main(void) {{
  bimamba_amp rec = {{0}};
  rec.scale = 65536.0f;
  printf("%d %d\\n", amp_step(0, 0, 4, 0, 0, 0, 0, 0, 0, 0, 0, &rec, 0, 0), bimamba_amp_update(0, 2.0, 0.5, 1, 0, 0));
  return 0;
}}
""")
    exe = tmp_path / "amp_host"
    lib = bm._lib.LIB_PATH
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", str(prog), "-o", str(exe), lib,
                           "-Wl,-rpath," + os.path.dirname(lib)])
    out = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    assert out == [-1, -1]


@pytest.mark.parametrize("kwargs", [dict(growth_factor=1.0), dict(growth_factor=0.5), dict(backoff_factor=1.0),
                                    dict(backoff_factor=2.0)])
def test_device_grad_scaler_refuses_what_torch_refuses(kwargs):
    with pytest.raises(AssertionError) as ours:
        bm.DeviceGradScaler(**kwargs)
    with pytest.raises(AssertionError) as theirs:
        torch.amp.GradScaler("cpu", **kwargs)      # "cuda" would disable itself on a machine without a GPU
    assert str(ours.value) == str(theirs.value)
    bm.DeviceGradScaler(enabled=False, **kwargs)   # a disabled scaler checks nothing, as torch's
    torch.amp.GradScaler("cpu", enabled=False, **kwargs)


def test_device_grad_scaler_defaults_state_dict_and_disabled_identity():
    ours, theirs = bm.DeviceGradScaler(), torch.amp.GradScaler("cpu")
    assert ours.state_dict() == theirs.state_dict() == {"scale": 65536.0, "growth_factor": 2.0, "backoff_factor": 0.5,
                                                        "growth_interval": 2000, "_growth_tracker": 0}
    custom = torch.amp.GradScaler("cpu", init_scale=8.0, growth_factor=3.0, backoff_factor=0.25, growth_interval=7)
    ours.load_state_dict(custom.state_dict())        # before the device record exists: held on the host
    assert ours.state_dict() == custom.state_dict()
    assert ours.get_scale() == 8.0
    with pytest.raises(RuntimeError, match="empty"):
        ours.load_state_dict({})
    off = bm.DeviceGradScaler(enabled=False)
    loss = torch.tensor(3.0)
    assert off.scale(loss) is loss and off.get_scale() == 1.0 and off.state_dict() == {} and not off.is_enabled()
