"""Host-independent CPU arithmetic for bit-exact comparisons on the CPU.  TEST INFRA.

By default torch picks CPU kernels by instruction set: oneDNN runs bf16 matmuls on AMX, AVX-512 or AVX2 code, ATen's
reductions and softmax use the widest vector type, and MKL dispatches fp32 GEMMs per CPU.  Each choice rounds differently
in the last bit, so a vector written on one CPU is not reproduced bit for bit on another.  A process started with
``ENV`` that calls ``apply()`` instead runs oneDNN-free, with ATen's portable kernels, MKL's reproducible code path and
one thread: the same results on every x86-64 host.  The golden generators under ``oracle/`` record what a test compares
bit for bit this way, and such tests, like those that compare two CPU runs bit for bit, run this way.
"""
import os

ENV = {"ATEN_CPU_CAPABILITY": "default", "MKL_CBWR": "COMPATIBLE", "OMP_NUM_THREADS": "1", "MKL_NUM_THREADS": "1"}


def active() -> bool:
    return all(os.environ.get(k) == v for k, v in ENV.items())


def apply():
    """Call in a process started with ``ENV`` (the variables are read when torch and MKL load)."""
    import torch
    assert active(), f"start the process with {ENV}"
    assert torch.backends.cpu.get_cpu_capability() == "DEFAULT", torch.backends.cpu.get_cpu_capability()
    torch.backends.mkldnn.enabled = False
    torch.set_num_threads(1)
