"""Kernel names, shared by the kernel-coverage tests: which kernels a call launched (torch.profiler) and which
instantiations the built library holds (cuobjdump -elf), both reduced to `base_kernel<template,args>` keys."""
import os
import re
import shutil
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "3d-multi-resolution-rcnn_b200", "lib", "libroi3d_b200.so")


def _demangle(names):
    if not names:
        return []
    cxxfilt = shutil.which("c++filt")
    assert cxxfilt, "c++filt (binutils) is needed to demangle kernel names"
    out = subprocess.run([cxxfilt], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return out.splitlines()


def kernel_key(name):
    """Base name plus template argument list with the spaces removed: `void roi3d::roi_align3d_fwd_cl_kernel<14, 7, 1,
    3>(roi3d::RoiParams)` -> `roi_align3d_fwd_cl_kernel<14,7,1,3>`.  None for a name that is not a `*_kernel`."""
    if name.startswith("_Z"):
        name = _demangle([name])[0]
    m = re.search(r"(\w+_kernel)\s*([<(]|$)", name)
    if m is None:
        return None
    key = m.group(1)
    if m.group(2) == "<":
        depth, i = 0, m.start(2)
        for j in range(i, len(name)):
            depth += {"<": 1, ">": -1}.get(name[j], 0)
            if depth == 0:
                key += name[i:j + 1]
                break
    return re.sub(r"\s+", "", key)


def launched_kernels(fn):
    """Run fn() under torch.profiler with CUDA activities and return the demangled names of the kernels that ran
    (memcpy / memset records excluded).  CUPTI sees every launch of the context, those of libroi3d_b200.so included."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA
             and not e.name.startswith(("Memcpy", "Memset", "cudaMem"))]
    assert names, "the profiler recorded no kernel: nothing would be checked"
    return names


def library_kernels(names):
    """Keys of the libroi3d_b200 kernels (namespace roi3d) among launched kernel names."""
    keys = [kernel_key(n) for n in names if "roi3d::" in n or n.startswith("_ZN5roi3d")]
    return {k for k in keys if k is not None}


def built_kernels(prefix):
    """Keys of the kernel instantiations in the built library whose name starts with `prefix`."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    assert os.path.exists(LIB), "%s is not built" % LIB
    assert os.path.exists(cuobjdump), "%s not found" % cuobjdump
    elf = subprocess.run([cuobjdump, "-elf", LIB], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(re.findall(r"\.text\.([A-Za-z0-9_$]+)", elf)))
    keys = {kernel_key(n) for n in _demangle(mangled)}
    return {k for k in keys if k is not None and k.startswith(prefix)}
