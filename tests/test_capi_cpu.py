"""CPU: the C-ABI library loads and exports every symbol include/b2s.h declares (no
compute calls without a GPU), and the product path fails loudly without CUDA."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def _declared():
    text = (ROOT / "include" / "b2s.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b2s_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from b200slam import _capi
    lib = ctypes.CDLL(str(_capi.lib_path()))
    names = _declared()
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/b2s.h but not exported"
    assert sorted(_capi.EXPORTS) == names
    assert _capi.load_library().b2s_abi_version() == _capi.ABI_VERSION


def test_header_constants_agree_with_host_and_oracle():
    from b200slam import _capi
    from oracle import hamming_oracle as ho
    text = (ROOT / "include" / "b2s.h").read_text()
    assert int(re.search(r"#define B2S_IDX_BITS (\d+)", text).group(1)) == _capi.IDX_BITS == ho.IDX_BITS
    assert int(re.search(r"#define B2S_SELECT_MAX_QUERIES (\d+)", text).group(1)) == _capi.SELECT_MAX_QUERIES
    assert _capi.NONE_KEY == int(ho.NONE_KEY)


def test_ratio_lut_is_the_oracle_lut():
    from b200slam.frontend import ratio_lut
    from oracle import hamming_oracle as ho
    for r in (0.6, 0.75, 0.8, 1.0, 0.37):
        np.testing.assert_array_equal(ratio_lut(r), ho.ratio_lut(r))


def test_sass_is_blackwell_native():
    """The built library carries sm_100a code, and the SHIPPED Hamming kernel itself — not just some kernel of the
    library — issues tcgen05.mma kind::i8 (SASS UTCIMMA), reads its accumulators from TMEM (LDTM), commits to
    mbarriers (UTCBAR) and stages operands with the TMA engine's bulk copies (UBLKCP); the tensor-core scoring kernel
    issues UTCHMMA; the POPC kernel keeps POPC + REDUX; the scoring kernel runs on packed FFMA2.  profiles/r02_sass.md is the committed listing (tools/sass_evidence.py)."""
    import shutil
    import subprocess
    from b200slam import _capi
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    out = subprocess.run(["cuobjdump", "-sass", str(_capi.lib_path())], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    funcs = {}
    cur = None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur is not None:
            funcs[cur].append(line)

    def body(*needles):
        hits = [k for k in funcs if all(n in k for n in needles)]
        assert hits, needles
        return "\n".join(funcs[hits[0]])
    k2s = body("hamming_knn2_i8s_kernel", "ILb1E")                  # <TOP2 = true>: the kNN-2 instantiation
    assert k2s.count("UTCIMMA") >= 18 and "LDTM" in k2s and "UTCBAR" in k2s and "UBLKCP" in k2s
    assert "VIMNMX3" in k2s and "VIADDMNMX" in k2s                  # the packed 16-bit key epilogue
    k2 = body("hamming_knn2_i8_kernel")
    assert k2.count("UTCIMMA") >= 18 and "LDTM" in k2
    k3t = body("ransac_score_tc_kernel")
    assert "UTCHMMA" in k3t and "LDTM" in k3t
    k1 = body("hamming_knn2_popc_kernel")
    assert "POPC" in k1 and "REDUX" in k1 and "UBLKCP" in k1
    k3h = body("ransac_score_hybrid_kernel")
    assert "DFMA" in k3h and k3h.count("FFMA2") >= 16 * 17              # packed fma.rn.f32x2: two correspondences per instruction


def test_product_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from b200slam import B2SError
    from integration.feature_pipeline_bridge import FeaturePipelineConfig, build_feature_pipeline
    from integration.pose_bridge import ransac_essential
    pipe = build_feature_pipeline(FeaturePipelineConfig())
    d = np.zeros((4, 32), np.uint8)
    with pytest.raises(B2SError):
        pipe.match(d, d)
    with pytest.raises(B2SError):
        ransac_essential(np.zeros((9, 2), np.float32), np.zeros((9, 2), np.float32), np.eye(3))


def test_product_never_imports_the_oracle():
    for base in (ROOT / "monocular-visual-slam_b200", ROOT / "integration"):
        for f in base.rglob("*.py"):
            src = f.read_text()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
