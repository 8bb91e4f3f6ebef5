"""oracle/build_ref_ext.py -- TEST INFRASTRUCTURE ONLY.

Compiles the REFERENCE's own PointNet++ CUDA extension (pointnet2._ext) from the sources where they lie under
/root/reference, into oracle/_ref/ (git-ignored; travels to the GPU box with the snapshot).  No reference source is copied
into this repository.  tools/make_golden_pn2_ref.py runs the resulting module on a GPU and stores the reference kernels'
outputs as tests/golden/pn2_ref.pt, against which tests/test_gpu_pn2_ref.py pins both the C restatement (oracle/pn2_oracle.c)
and the sam6d_b200 kernels; bench.py times it next to ours when it is present.

The reference's setup.py does not build as shipped (relative include_dirs, PEM/model/pointnet2/setup.py:23), so this is our
own recipe: torch.utils.cpp_extension.load with an absolute include path and an sm_100 target.
"""
import glob
import os

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
SRC = "/root/reference/SAM-6D/Pose_Estimation_Model/model/pointnet2/_ext_src"
NAME = "pointnet2_ref_ext"


def so_path():
    hits = glob.glob(os.path.join(OUT, NAME + "*.so"))
    return hits[0] if hits else None


def build():
    if so_path():
        return so_path()
    if not os.path.isdir(SRC):
        raise RuntimeError("reference sources not present (this only builds in the dev container)")
    os.makedirs(OUT, exist_ok=True)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
    from torch.utils.cpp_extension import load
    srcs = sorted(glob.glob(os.path.join(SRC, "src", "*.cpp")) + glob.glob(os.path.join(SRC, "src", "*.cu")))
    load(name=NAME, sources=srcs, extra_include_paths=[os.path.join(SRC, "include")], build_directory=OUT,
         extra_cflags=["-O2"], extra_cuda_cflags=["-O2"], verbose=False, is_python_module=False)
    return so_path()


def load_module():
    """import the prebuilt reference extension (GPU box: only the .so exists)"""
    path = so_path()
    if path is None:
        return None
    import importlib.util
    import torch  # noqa: F401  (the extension links against libtorch)
    spec = importlib.util.spec_from_file_location(NAME, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    print(build())
