"""B200-native device plugin + node labeller core (host-side mirror of the reference's Go packages).

Python here is the host language above the C ABI (include/b200dp.h) because the Go
toolchain is absent from the build image; every module mirrors one reference package:

    amdgpu     <- internal/pkg/amdgpu          plugin   <- internal/pkg/plugin + cmd/k8s-device-plugin
    allocator  <- internal/pkg/allocator       exporter <- internal/pkg/exporter
    labeller   <- cmd/k8s-node-labeller        context  <- the backend handle (kfd: / cuda:)

All arithmetic happens in libb200dp.so (C++/CUDA); nothing here imports `oracle/`.
"""
from . import _native  # noqa: F401  (raises if libb200dp.so is missing: no fallback)
from . import allocator, amdgpu, exporter, labeller, plugin, synth, v1beta1  # noqa: F401
from .context import Context, compute_expected  # noqa: F401

__all__ = ["Context", "amdgpu", "allocator", "plugin", "exporter", "labeller"]
