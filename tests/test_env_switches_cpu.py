"""CPU check of the library's environment switches: the only OB200_* variables the CUDA sources read are the multi-GPU and
operational settings below. Every other choice is fixed in the code, so no untested kernel variant can be selected from the
environment."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "clima-oceananigans.jl_b200", "csrc")

ALLOWED = {
    "OB200_NO_P2P", "OB200_LINK_TIMEOUT_S", "OB200_QUIET", "OB200_NCCL_BARRIER", "OB200_NO_PEER_HALO",
    "OB200_NO_HALO_OVERLAP", "OB200_NO_FFT_DTMA", "OB200_FFT_BULK_A2A", "OB200_FFT_YSPLIT", "OB200_FFT_YBLOCKS",
}


def read_names():
    pat = re.compile(r'\b(?:getenv|env_int)\s*\(\s*"(OB200_\w*)"')
    names = set()
    for f in sorted(os.listdir(CSRC)):
        if f.endswith((".cu", ".cuh", ".h", ".cpp")):
            names |= set(pat.findall(open(os.path.join(CSRC, f)).read()))
    return names


def test_only_multi_gpu_and_operational_switches_remain():
    assert read_names() == ALLOWED
