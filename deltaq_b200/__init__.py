"""deltaq_b200 -- B200 (sm_100a) suffix sorter and bsdiff match engine behind DeltaQ's ISuffixSort contract.

Only what the hot path needs: csrc/ (CUDA kernels + C ABI, built into libdeltaq_cuda.so), the host-side
mirror of the reference's provider / Diff interface, and the synthetic workloads of BASELINE.json.
There is no CPU fallback: every entry point raises when libdeltaq_cuda.so or a CUDA device is missing.
"""
from .suffix_sort import CudaSuffixSort, SuffixArrayOwner, SuffixArraysOwner  # noqa: F401

__all__ = ["CudaSuffixSort", "SuffixArrayOwner", "SuffixArraysOwner"]
