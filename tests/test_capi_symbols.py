"""CPU test: libsxgpu.so loads, and exports every function include/sxgpu.h declares -- no
compute calls (there is no GPU here)."""
import ctypes as C
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def declared_functions():
    text = (ROOT / "include" / "sxgpu.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sxgpu_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_hot_path():
    names = declared_functions()
    for must in ("sxgpu_convert_rx_buffer", "sxgpu_convert_tx_buffer", "sxgpu_convert_rx_buffer_host",
                 "sxgpu_convert_tx_buffer_host", "sxgpu_convert_rx_batch", "sxgpu_convert_tx_batch", "sxgpu_init"):
        assert must in names


def test_library_exports_every_declared_symbol():
    from sxxcvr_b200 import capi
    lib = capi.load_library()
    for name in declared_functions():
        assert hasattr(lib, name), f"{name} declared in include/sxgpu.h but not exported"
        assert name in capi.SIGNATURES, f"{name} has no ctypes signature in sxxcvr_b200/capi.py"
    assert set(capi.SIGNATURES) == set(declared_functions())
    assert lib.sxgpu_abi_version() == 1
    assert lib.sxgpu_strerror(-3) == b"no usable sm_100 device"


def test_library_is_sm100a_only_and_has_no_cpu_path():
    from sxxcvr_b200 import capi
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", str(capi.library_path())], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump not available")
    archs = set(re.findall(r"sm_\d+a?", out.stdout))
    assert archs == {"sm_100a"}, archs


def test_forced_build_links_each_target_once_and_leaves_none_stale(tmp_path, monkeypatch):
    """build() forces every target.  Each must be linked once, after what it links against: a
    target left older than a dependency is relinked in the tree by the next load, which fails
    where the tree is read-only.  The compiler is replaced by a recorder that writes each output
    with a strictly later time stamp."""
    import os
    import time
    from sxxcvr_b200 import _build
    for name in ("GPU_LIB", "SOAPY_LIB", "EXAMPLE_BIN", "HOOK_EXAMPLE_LIB"):
        monkeypatch.setattr(_build, name, tmp_path / getattr(_build, name).name)
    monkeypatch.setattr(_build, "LIB", tmp_path)
    linked, clock = [], [time.time() + 10]

    def record(cmd):
        out = Path(cmd[cmd.index("-o") + 1])
        out.write_bytes(b"")
        clock[0] += 1
        os.utime(out, (clock[0], clock[0]))
        linked.append(out.name)

    monkeypatch.setattr(_build, "_run", record)
    monkeypatch.setattr(_build, "_find_nvcc", lambda: "nvcc")
    _build.build_all(force=True)
    assert sorted(linked) == sorted(p.name for p in (_build.GPU_LIB, _build.SOAPY_LIB, _build.EXAMPLE_BIN,
                                                     _build.HOOK_EXAMPLE_LIB))
    _build.build_all()
    assert len(linked) == 4, linked[4:]


def test_init_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from sxxcvr_b200 import Context, SxGpuError
    with pytest.raises(SxGpuError) as e:
        Context(0)
    assert e.value.code == -3


def test_product_does_not_link_the_oracle():
    """The oracle is test infrastructure: nothing under sxxcvr_b200/ may reference it."""
    for path in (ROOT / "sxxcvr_b200").rglob("*"):
        if path.suffix in (".py", ".cpp", ".hpp", ".h", ".cu", ".cuh"):
            text = path.read_text()
            for needle in ("sx_oracle.h", "sxo_", "sxref_", "dlopen", "libsx_oracle"):
                assert needle not in text, (path, needle)
    import subprocess
    for lib in (ROOT / "sxxcvr_b200" / "lib").glob("*.so"):
        needed = subprocess.run(["readelf", "-d", str(lib)], capture_output=True, text=True).stdout
        assert "oracle" not in needed and "sx_ref" not in needed, lib
