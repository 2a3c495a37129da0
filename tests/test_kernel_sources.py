"""CPU: the tcgen05 kernels share one copy of their device primitives and of each operand format."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "fastspeech2_b200", "csrc")
PRIMITIVES = "tc_ptx.cuh"


def _sources():
    out = {}
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh")):
            txt = open(os.path.join(CSRC, f)).read()
            out[f] = re.sub(r"//[^\n]*", "", txt)   # comments may name the instructions
    return out


def test_tensor_core_ptx_lives_only_in_the_primitives_header():
    mnemonic = re.compile(r"\b(tcgen05\.|mbarrier\.|cp\.async\.bulk|cp\.reduce\.async\.bulk|elect\.sync|fence\.mbarrier_init)")
    found = {}
    for f, txt in _sources().items():
        for stmt in re.findall(r"\basm\s*(?:volatile\s*)?\((.*?)\);", txt, flags=re.S):
            if mnemonic.search(stmt):
                found.setdefault(f, []).append(mnemonic.search(stmt).group(1))
    assert PRIMITIVES in found
    assert set(found) == {PRIMITIVES}, {f: m for f, m in found.items() if f != PRIMITIVES}


def test_fused_kernels_do_not_include_the_conv_kernel():
    src = _sources()
    for f in ("resstack_fused.cu", "attention_fused.cu"):
        includes = re.findall(r'#include\s+"([^"]+)"', src[f])
        assert "conv_tc_kernel.cuh" not in includes, f


def test_operand_formats_are_defined_once():
    src = _sources()
    for name in ("TC_F8_LO_SCALE", "TC_F8_HI_SCALE", "KV_WSCALE", "TC_HDR", "kv_tile_stride"):
        defs = [f for f, txt in src.items() if re.search(r"\b(?:constexpr\s+\w+|long long)\s+" + name + r"\b", txt)]
        assert len(defs) == 1, (name, defs)
    for stale in ("AT_WSCALE", "AF_WSCALE", "AT_HDR", "at_tile_stride", "af_tile_stride"):
        assert not any(re.search(r"\b" + stale + r"\b", txt) for txt in src.values()), stale
