"""Build the reference's own pvcnn and Chamfer CUDA extensions into oracle/_ref/ (TEST INFRASTRUCTURE ONLY).

The reference's point-op kernels (third_party/pvcnn/functional/src/**/*.cu, bound in
src/bindings.cpp:10-37) compile from their own 13 source files with nothing but torch's
headers, so they are compiled *from where they lie* under /root/reference with a recipe of our
own (the reference's recipe is a JIT `load()` inside backend.py:8-27 that writes next to the
sources, which are read-only here).  No reference source is copied into this repo; only the
built `_pvcnn_backend.so` lands in oracle/_ref/ (git-ignored, shipped to the GPU box).

Its outputs on the GPU tests' inputs are the ground truth stored in tests/golden/ref_*.npz by
tests/golden/make_golden_ref_kernels.py, above all for the index-producing ops (FPS, ball query,
3-NN, voxel indices) -- their results depend on nvcc's FMA contraction, which a CPU restatement can
only approximate.  bench.py's `parity` and `gpu_baseline` legs use it where it was built; the
product path never does.

The Chamfer extension (third_party/ChamferDistancePytorch/chamfer3D/{chamfer_cuda.cpp,
chamfer3D.cu}, JIT-loaded by dist_chamfer_3D.py:12-16 with default flags) is built the same way
into oracle/_ref/chamfer_3D.so: ground truth for lion_chamfer_forward (distances bit-exact,
indices exact).

The approximate-EMD extension (third_party/PyTorchEMD/cuda/{emd.cpp,emd_kernel.cu}) is built into
oracle/_ref/emd_ext.so with oracle/shim/ on the include path (it supplies the removed THC header the
kernel source still includes): ground truth for lion_emd_approx.

Run:  python oracle/build_ref.py          (no GPU needed; ~4 min)
"""
import os
import sys

REF_SRC = "/root/reference/third_party/pvcnn/functional/src"
OUT_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
SOURCES = [
    "ball_query/ball_query.cpp", "ball_query/ball_query.cu",
    "grouping/grouping.cpp", "grouping/grouping.cu",
    "interpolate/neighbor_interpolate.cpp", "interpolate/neighbor_interpolate.cu",
    "interpolate/trilinear_devox.cpp", "interpolate/trilinear_devox.cu",
    "sampling/sampling.cpp", "sampling/sampling.cu",
    "voxelization/vox.cpp", "voxelization/vox.cu",
    "bindings.cpp",
]


def build(verbose=False):
    so = os.path.join(OUT_DIR, "_pvcnn_backend.so")
    if os.path.exists(so):
        return so
    if not os.path.isdir(REF_SRC):
        return None  # GPU box: only the prebuilt file is used
    os.makedirs(OUT_DIR, exist_ok=True)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")
    from torch.utils.cpp_extension import load
    load(name="_pvcnn_backend",
         sources=[os.path.join(REF_SRC, s) for s in SOURCES],
         extra_cflags=["-O3", "-std=c++17"],       # backend.py:10
         build_directory=OUT_DIR, verbose=verbose, is_python_module=False)
    return so if os.path.exists(so) else None


CHAMFER_SRC = "/root/reference/third_party/ChamferDistancePytorch/chamfer3D"


def build_chamfer(verbose=False):
    so = os.path.join(OUT_DIR, "chamfer_3D.so")
    if os.path.exists(so):
        return so
    if not os.path.isdir(CHAMFER_SRC):
        return None
    os.makedirs(OUT_DIR, exist_ok=True)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")
    from torch.utils.cpp_extension import load
    load(name="chamfer_3D",
         sources=[os.path.join(CHAMFER_SRC, "chamfer_cuda.cpp"), os.path.join(CHAMFER_SRC, "chamfer3D.cu")],
         build_directory=OUT_DIR, verbose=verbose, is_python_module=False)       # dist_chamfer_3D.py:12-16: default flags
    return so if os.path.exists(so) else None


def load_chamfer():
    import importlib.util
    import torch  # noqa: F401
    so = os.path.join(OUT_DIR, "chamfer_3D.so")
    if not os.path.exists(so):
        return None
    spec = importlib.util.spec_from_file_location("chamfer_3D", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


EMD_SRC = "/root/reference/third_party/PyTorchEMD/cuda"


def build_emd(verbose=False):
    """third_party/PyTorchEMD/backend.py:10-19 JIT-loads cuda/emd.cpp + cuda/emd_kernel.cu with -O3 -std=c++17;
    the kernel source includes the long-removed <THC/THC.h>, which oracle/shim/ supplies (two macros)."""
    so = os.path.join(OUT_DIR, "emd_ext.so")
    if os.path.exists(so):
        return so
    if not os.path.isdir(EMD_SRC):
        return None
    os.makedirs(OUT_DIR, exist_ok=True)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")
    from torch.utils.cpp_extension import load
    shim = os.path.join(os.path.dirname(os.path.abspath(__file__)), "shim")
    load(name="emd_ext", sources=[os.path.join(EMD_SRC, "emd.cpp"), os.path.join(EMD_SRC, "emd_kernel.cu")],
         extra_cflags=["-O3", "-std=c++17"], extra_include_paths=[shim],
         build_directory=OUT_DIR, verbose=verbose, is_python_module=False)
    return so if os.path.exists(so) else None


def load_emd():
    import importlib.util
    import torch  # noqa: F401
    so = os.path.join(OUT_DIR, "emd_ext.so")
    if not os.path.exists(so):
        return None
    spec = importlib.util.spec_from_file_location("emd_ext", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_ref():
    """Import oracle/_ref/_pvcnn_backend.so (needs a GPU to *run* its functions)."""
    import importlib.util
    import torch  # noqa: F401  (libtorch symbols must be loaded first)
    so = os.path.join(OUT_DIR, "_pvcnn_backend.so")
    if not os.path.exists(so):
        return None
    spec = importlib.util.spec_from_file_location("_pvcnn_backend", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv))
    print(build_chamfer(verbose="-v" in sys.argv))
    print(build_emd(verbose="-v" in sys.argv))
