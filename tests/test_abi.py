"""The C-ABI library builds, loads on a CPU-only host and exports every symbol include/tokenhmr_b200.h
declares (no compute calls here)."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def _declared():
    text = (ROOT / "include" / "tokenhmr_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(thmr_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported_and_bound(built_lib):
    from tokenhmr_b200._lib import SIGNATURES
    names = _declared()
    assert len(names) >= 25
    for n in names:
        assert hasattr(built_lib, n), f"{n} declared in the header but not exported"
        assert n in SIGNATURES, f"{n} has no ctypes signature"
    assert set(SIGNATURES) == set(names)


def test_version_and_error_string(built_lib):
    assert built_lib.thmr_abi_version() >= 2
    assert isinstance(built_lib.thmr_last_error(), bytes)


def test_struct_layouts_match_header_field_counts():
    """Cheap guard against header / ctypes drift: field names of every mirrored struct appear in the header."""
    from tokenhmr_b200 import _lib
    text = (ROOT / "include" / "tokenhmr_b200.h").read_text()
    for cls in (_lib.SmplDesc, _lib.Config, _lib.VitBlock, _lib.DecLayer, _lib.MixerBlock, _lib.Conv, _lib.Weights,
                _lib.Outputs, _lib.PreprocCfg, _lib.TokConv, _lib.TokEncoderDesc):
        for name, _ in cls._fields_:
            assert re.search(rf"\b{name}\b", text), f"{cls.__name__}.{name} not in header"
    assert ctypes.sizeof(_lib.Outputs) == 12 * ctypes.sizeof(ctypes.c_void_p)


def test_header_is_plain_c_and_struct_sizes_match_ctypes(tmp_path):
    """include/tokenhmr_b200.h must compile as C (the boundary is a C ABI) and every struct mirrored in _lib.py must
    have the size the C compiler gives it."""
    import shutil
    import subprocess
    from tokenhmr_b200 import _lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no C compiler")
    pairs = [("thmr_smpl_desc", _lib.SmplDesc), ("thmr_config", _lib.Config), ("thmr_vit_block", _lib.VitBlock),
             ("thmr_dec_layer", _lib.DecLayer), ("thmr_mixer_block", _lib.MixerBlock), ("thmr_conv", _lib.Conv),
             ("thmr_weights", _lib.Weights), ("thmr_outputs", _lib.Outputs), ("thmr_preproc_cfg", _lib.PreprocCfg),
             ("thmr_tok_conv", _lib.TokConv), ("thmr_tok_encoder_desc", _lib.TokEncoderDesc)]
    src = tmp_path / "sizes.c"
    body = "".join(f'  printf("%s %zu\\n", "{n}", sizeof({n}));\n' for n, _ in pairs)
    src.write_text(f'#include <stdio.h>\n#include "{ROOT / "include" / "tokenhmr_b200.h"}"\nint main(void) {{\n{body}  return 0;\n}}\n')
    exe = tmp_path / "sizes"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(src)], check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    sizes = dict(zip(out[0::2], map(int, out[1::2])))
    for name, cls in pairs:
        assert sizes[name] == ctypes.sizeof(cls), f"{name}: C {sizes[name]} vs ctypes {ctypes.sizeof(cls)}"


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from tokenhmr_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", tmp_path / "nope.so")
    with pytest.raises(_lib.ThmrError, match="no non-CUDA fallback"):
        _lib.lib()


def test_engine_refuses_cpu_device():
    from tokenhmr_b200 import _lib
    from tokenhmr_b200.config import tiny_config
    from tokenhmr_b200.engine import TokenHMREngine
    with pytest.raises(_lib.ThmrError, match="no CPU fallback"):
        TokenHMREngine(tiny_config(), {}, {}, device="cpu")


def test_product_never_imports_the_oracle():
    for f in (ROOT / "tokenhmr_b200").rglob("*.py"):
        src = f.read_text()
        assert "import oracle" not in src and "from oracle" not in src, f


def test_library_reads_only_the_known_environment_variables():
    """Every getenv() of the native library selects something a caller relies on: THMR_VQ_SCREEN and THMR_SKIN_THREADS
    pick between two timed schedules, THMR_NCCL_LIB locates a library.  A new switch has to be added here on purpose."""
    names = set()
    for f in sorted((ROOT / "tokenhmr_b200" / "csrc").glob("*.cu*")):
        names.update(re.findall(r'getenv\(\s*"([^"]+)"', f.read_text()))
    assert names == {"THMR_VQ_SCREEN", "THMR_SKIN_THREADS", "THMR_NCCL_LIB"}


def test_vq_workspace_covers_both_schedules(built_lib):
    """thmr_vq_workspace_bytes is pure arithmetic (no CUDA call): it covers BOTH schedules of thmr_vq_argmin (the single exact
    pass needs a Q x 3D fp16 split operand; the screened one a 131072-row fp16 chunk, a 262144-row exact-pass round and the row
    queue), so that switching THMR_VQ_SCREEN never invalidates a caller's buffer, and it never shrinks when Q grows."""
    K, D = 2048, 256
    small = built_lib.thmr_vq_workspace_bytes(960, K, D)
    assert small >= 960 * 3 * D * 2 + K * 3 * D * 2
    prev = 0
    for Q in (960, 8192, 40960, 262144, 1_000_000, 4_000_000):
        n = built_lib.thmr_vq_workspace_bytes(Q, K, D)
        assert n >= prev and n % 1024 == 0
        prev = n
    assert built_lib.thmr_vq_workspace_bytes(1_000_000, K, D) >= 1_000_000 * 3 * D * 2 + 1_000_000 * 4     # exact layout covered
    assert built_lib.thmr_vq_workspace_bytes(1_000_000, K, D) >= 131072 * D * 2 + 262144 * 3 * D * 2 + 1_000_000 * 8  # screened
    assert built_lib.thmr_abi_version() >= 5          # thmr_config::concurrent
