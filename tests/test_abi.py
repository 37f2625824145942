"""The C-ABI library loads without a GPU and exports every symbol include/dadd_b200.h declares (no compute calls)."""

import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "dadd_b200.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dadd_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    from progressive_stable_diffusion_b200 import _lib
    return _lib


def test_header_declares_the_expected_entry_points():
    names = _declared()
    for n in ("dadd_ddim_step", "dadd_ddim_step_table", "dadd_step_begin", "dadd_groupnorm_fwd", "dadd_layernorm_fwd",
              "dadd_geglu_fwd", "dadd_add_layernorm_fwd", "dadd_groupnorm_cat_fwd", "dadd_groupnorm_cat_supported",
              "dadd_upsample_nearest2x_fwd", "dadd_ff_geglu_fwd", "dadd_quick_gelu_fwd", "dadd_linear_fwd", "dadd_linear_supported", "dadd_bias_residual_fwd", "dadd_groupnorm_workspace_bytes",
              "dadd_cross_attn_fwd", "dadd_self_attn_fwd", "dadd_purifier_attn_fwd",
              "dadd_purifier_gate_ln_fwd", "dadd_aoe_interp_fwd", "dadd_image_post_fwd", "dadd_last_error",
              "dadd_abi_version", "dadd_launch_count", "dadd_reset_launch_count"):
        assert n in names, n


def test_library_exports_every_declared_symbol(lib):
    cdll = ctypes.CDLL(lib.LIB_PATH)
    for n in _declared():
        assert hasattr(cdll, n), f"{n} declared in dadd_b200.h but not exported by libdadd_b200.so"


def test_ctypes_table_covers_the_header(lib):
    helpers = {"dadd_last_error", "dadd_abi_version", "dadd_launch_count", "dadd_reset_launch_count"}
    assert set(lib.SIGNATURES) == set(_declared()) - helpers
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for name, args in lib.SIGNATURES.items():
        m = re.search(r"\b" + name + r"\s*\((.*?)\)\s*;", src, flags=re.S)
        assert m, name
        assert len([a for a in m.group(1).split(",") if a.strip()]) == len(args), name


def test_abi_version_and_error_channel(lib):
    l = lib.load()
    assert l.dadd_abi_version() == lib.ABI_VERSION
    # argument validation happens before any CUDA call, so it is testable without a GPU
    rc = l.dadd_groupnorm_fwd(None, None, None, None, 0, None, 1, 320, 64, 32, 1e-5, 1, 1, 1, None, 0, None)
    assert rc != 0 and b"dadd_groupnorm_fwd" in l.dadd_last_error()
    rc = l.dadd_cross_attn_fwd(1, 320, 1, 1, 1, 320, 1, 8, 64, 41, 16, 3, 1, 0.1, 1, 0, None)
    assert rc != 0 and b"d % 8" in l.dadd_last_error()


def test_missing_library_fails_loudly(lib, monkeypatch):
    monkeypatch.setattr(lib, "_lib", None)
    monkeypatch.setattr(lib, "LIB_PATH", "/nonexistent/libdadd_b200.so")
    with pytest.raises(lib.DaddError):
        lib.load()


def test_argument_validation_of_the_newer_entry_points(lib):
    """Every entry point validates shapes / alignment before touching CUDA, so the error channel is testable without a GPU."""
    l = lib.load()
    err = lambda: l.dadd_last_error().decode()
    assert l.dadd_linear_supported(1024, 320, 320) == 1 and l.dadd_linear_supported(1024, 96, 320) == 0
    assert l.dadd_linear_supported(1024, 320, 324) == 0                     # K % 8
    assert l.dadd_linear_fwd(16, 16, None, None, 16, 128, 96, 320, 1, None) != 0 and "N % 64 == 0" in err()
    assert l.dadd_linear_fwd(None, 16, None, None, 16, 128, 320, 320, 1, None) != 0 and "dadd_linear_fwd" in err()
    assert l.dadd_ff_geglu_fwd(16, 16, 16, 16, 128, 320, 1000, 1, None) != 0 and "inner % 128" in err()
    assert l.dadd_ff_geglu_fwd(16, 16, 16, 16, 128, 320, 1280, 0, None) != 0 and "dtype16_ok" in err()      # fp32 not taken
    assert l.dadd_self_attn_fwd(16, 16, 16, 600, 600, 600, 16, 200, 1, 1, 64, 200, 0.1, 1, 0, None) != 0 and "wide" in err()   # d = 200
    assert l.dadd_groupnorm_select(1) == 0 and l.dadd_groupnorm_select(0) == 1
    assert l.dadd_ema_update(None, 16, 64, 0.999, 0, None) != 0 and "dadd_ema_update" in err()
    assert l.dadd_ema_update(16, 16, 64, 1.5, 0, None) != 0 and "decay" in err()
    assert l.dadd_ema_update(16, 24, 64, 0.9, 0, None) != 0                                           # 16-byte alignment
    assert l.dadd_adamw_step_dev(16, 16, 16, 16, 64, 1e-4, 0.9, 0.999, 1e-8, 0.01, None, None, None) != 0 and "dev_state" in err()
    assert l.dadd_sumsq(None, 64, 16, 1, None) != 0 and "n == 0" in err()      # only an empty buffer may come without an address
    assert l.dadd_sumsq(24, 64, 16, 1, None) != 0 and "dadd_sumsq" in err()    # 16-byte alignment
    assert l.dadd_groupnorm_cat_supported(4, 640, 320, 1024, 32, 1) == 1
    assert l.dadd_groupnorm_cat_supported(4, 644, 320, 1024, 32, 1) == 0    # C1 % 8
    assert l.dadd_groupnorm_cat_supported(4, 640, 320, 1024, 32, 0) == 0    # fp32
    assert l.dadd_groupnorm_cat_fwd(16, 644, 16, 320, 16, 16, None, 0, 16, 4, 1024, 32, 1e-5, 1, 1, None, 0, None) != 0
    assert "dadd_groupnorm_cat_fwd" in err()
    assert l.dadd_upsample_nearest2x_fwd(16, 16, 1, 8, 8, 12, 1, None) != 0 and "C % 8" in err()
    assert l.dadd_quick_gelu_fwd(16, 16, 12, 1, None) != 0 and "n % 8" in err()
    assert l.dadd_cross_attn_fwd(16, 320, 16, 16, 16, 320, 1, 8, 64, 40, 16, 3, 16, 0.1, 1, 2, None) != 0 and "impl = 2" in err()
    assert l.dadd_add_layernorm_fwd(16, 16, None, 16, 16, 16, 16, 4, 320, 1e-5, 1, None) != 0            # sum_bias without sum_out
    assert l.dadd_purifier_attn_fwd(16, 16, 16, 16, 1, 16, 100000, 768, 8, None) != 0 and "shared memory" in err()


def test_shipped_library_is_blackwell_native(lib):
    """The hot kernels of the built library carry the sm_100a instructions the design claims (cuobjdump -sass, no GPU needed):
    tcgen05 MMAs (UTCHMMA) with TMEM loads / stores and TMA tensor loads / stores in the self- and cross-attention cores, the
    feed-forward GEGLU GEMM and the linear GEMM (whose CTA-pair form adds `.2CTA` MMAs), and no kernel built for another arch."""
    import shutil
    import subprocess
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    lib.load()
    sass = subprocess.run(["cuobjdump", "-sass", lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert "arch = sm_100a" in sass
    per = {}
    name, arch = None, None
    for line in sass.splitlines():
        a = re.search(r"arch = (sm_\w+)", line)
        if a:
            arch = a.group(1)
        m = re.search(r"Function : (\S+)", line)
        if m:
            assert arch == "sm_100a", (m.group(1), arch)      # (the link step's empty default-arch stub holds no function)
            name = m.group(1)
            per[name] = line[:0]
            continue
        if name and re.search(r"UTCHMMA|UTMALDG|UTMASTG|LDTM|STTM|UBLKCP", line):
            per[name] += re.search(r"(UTCHMMA(\.2CTA)?|UTMALDG|UTMASTG|LDTM|STTM|UBLKCP)", line).group(1) + " "
    def kernels(tag):
        return [v for k, v in per.items() if tag in k]
    for tag in ("self_attn_tc_kernel", "cross_attn_tc_kernel", "ff_geglu_kernel", "linear_kernel"):
        ks = kernels(tag)
        assert ks and all("UTCHMMA" in v and "UTMALDG" in v and "LDTM" in v for v in ks), tag
    assert any("UTCHMMA.2CTA" in v for v in kernels("linear_kernel")), "the CTA-pair linear GEMM lost its cta_group::2 MMAs"
    assert all("STTM" in v for v in kernels("self_attn_tc_kernel")) and all("UTMASTG" in v for v in kernels("ff_geglu_kernel"))
    assert all("UTMALDG" in v and "UTMASTG" in v for v in kernels("gn_stream_kernel")) and kernels("gn_cluster_kernel")
