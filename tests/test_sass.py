"""The built library really contains the sm_100a features DESIGN.md claims (checked in the SASS, no GPU needed)."""
import functools
import re
import shutil
import subprocess

import pytest

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


@functools.lru_cache(maxsize=1)
def _sass() -> str:
    import cudavideostream_b200 as cvs
    try:
        return subprocess.run([CUOBJDUMP, "-sass", cvs.library_path()], capture_output=True, text=True, check=True).stdout
    except (OSError, subprocess.CalledProcessError) as e:
        pytest.skip(f"cuobjdump unavailable: {e}")


def _function(name_regex: str) -> str:
    blocks = re.split(r"(?=\n\s*Function : )", _sass())
    hit = [b for b in blocks if re.search(r"Function : \S*" + name_regex, b)]
    assert hit, f"no kernel matching {name_regex} in the library"
    return hit[0]


def test_library_is_sm_100a_only():
    archs = set(re.findall(r"arch = (sm_\w+)", _sass()))
    assert archs == {"sm_100a"}, archs


def test_stream_kernel_uses_tma_bulk_copies_and_byte_simd():
    k = _function(r"k_streamILi0ELb0EE")             # k_stream<0, false>
    assert "UBLKCP" in k, "the frame ingest must be a TMA bulk copy (cp.async.bulk)"
    assert "SYNCS" in k, "mbarrier (SYNCS.*) expected next to the bulk copy"
    assert k.count("VABSDIFF4") >= 24, "one byte-SIMD absolute difference per word of the 96-byte chunk"
    assert "REDUX" in k, "warp totals by redux.sync"
    assert "HMMA" not in k and "UTC" not in k, "byte work: no tensor-core instructions expected"


def test_no_kernel_spills_in_the_hot_variants():
    # local-memory traffic (LDL/STL) in the default-mode stream kernels would mean register spills
    for name in (r"k_streamILi0ELb0EE", r"k_stream_wsILi0ELb0EE"):
        k = _function(name)
        assert not re.search(r"\b(LDL|STL)\b", k), f"{name} spills to local memory"


def test_noise_filter_is_fma_in_fixed_order():
    # every k_conv_strip<K, NONNEG, WB> launch_conv can pick: WB words (4*WB bytes) per thread
    for K, nonneg, wb in ((3, True, 2), (3, False, 2), (3, True, 1), (3, False, 1), (5, True, 1), (5, False, 1)):
        name = r"k_conv_stripILi%dELb%dELi%dE" % (K, int(nonneg), wb)
        k = _function(name)
        # packed fp32 (sm_100): one FFMA2 carries the same tap of two neighbouring output bytes, each half rounded like FFMA
        assert len(re.findall(r"\bFFMA2\b", k)) == 8 * 2 * wb * K * K, f"{name}: 8 rows x 2*WB byte pairs x K*K taps, one FFMA2 each"
        assert not re.search(r"\bFFMA\b", k), f"{name}: no scalar FFMA left"
        assert re.search(r"\bFADD2\b", k), f"{name}: byte -> float is packed too"
        if nonneg:
            assert re.search(r"\bFADD2\.RZ\b", k), f"{name}: truncation is packed too"
            assert "F2I" not in k, f"{name}: non-negative weights truncate with FADD.RZ, not F2I"
        assert not re.search(r"\b(LDL|STL)\b", k), f"{name}: the row window must stay in registers"
