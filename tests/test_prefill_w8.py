"""The int8 prompt GEMM (kllm_gemm_w8) as compiled for sm_100a, checked on the CPU from its SASS: it runs on
the 5th-generation tensor cores (tcgen05.mma.kind::i8 -> UTCIMMA), is fed by TMA tensor loads (UTMALDG) and
reads its accumulators back from tensor memory (tcgen05.ld -> LDTM); the 64 per-token running sums of its
epilogue stay in registers (no stack frame, next to no local memory)."""
import re
import subprocess

from kuiperllama_b200 import build as kbuild

KERNEL = "_ZN4kllm2tc14gemm_w8_kernelE14CUtensorMap_stS1_PKfS3_Pfiiii"
QUANTISER = "_ZN4kllm2tc23quantize_w8_rows_kernelEPKfPhPfiii"


def _sass(name):
    return subprocess.run(["cuobjdump", "-sass", "-fun", name, str(kbuild.LIB)], capture_output=True, text=True,
                          check=True).stdout


def _usage():
    res = subprocess.run(["cuobjdump", "-res-usage", str(kbuild.LIB)], capture_output=True, text=True,
                         check=True).stdout
    return {m.group(1): (int(m.group(2)), int(m.group(3)))
            for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", res)}


def test_gemm_w8_runs_on_kind_i8_tensor_cores(kllm_lib):
    sass = _sass(KERNEL)
    for op in ("UTCIMMA", "UTMALDG", "LDTM"):
        assert re.search(rf"\b{op}\b", sass), f"{op} missing from {KERNEL}"
    assert not re.search(r"\b(UTCHMMA|UTCQMMA|HMMA|IMMA)\b", sass), "another MMA flavour in the int8 GEMM"


def test_gemm_w8_keeps_its_sums_in_registers(kllm_lib):
    usage = _usage()
    for name in (KERNEL, QUANTISER):
        assert name in usage, sorted(k for k in usage if "w8" in k)
        regs, stack = usage[name]
        assert stack <= 16, f"{name}: {stack} bytes of stack"
        local = len(re.findall(r"\b(?:LDL|STL)(?:\.\S+)?\b", _sass(name)))
        assert local <= 4, f"{name}: {local} local-memory instructions"
