"""Run the UNMODIFIED reference checkout (staged by tools/stage_reference.sh into baseline/_ref/HairFastGAN) in this
image: import-time stand-ins for the packages the image lacks (SURVEY Appendix D: clip, dlib, face_alignment, lpips,
matplotlib, gdown, addict, torchmetrics -> baseline/stubs/), the prebuilt JIT-extension cache, the working directory
the reference's relative paths assume (`pretrained_models/...`, `models/sean_codes/styles_test/...`), and -- optionally
-- this package's overlay (hairfastgan_b200.install) on top.

    import baseline.refenv as refenv
    refenv.activate(overlay=True)                 # or overlay=False: the stock reference (its cuDNN + JIT kernels)
    from hair_swap import HairFast, get_parser    # the reference's own file, unchanged

One process = one mode (the reference's modules are cached in sys.modules).  Nothing here is product code: it is the
harness of baseline/run_swap.py, of `bench.py`'s full-swap / reference legs and of tools/dryrun_swap_cpu.py.
"""
from __future__ import annotations

import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
STUBS = os.path.join(HERE, "stubs")
REF_DIR = os.path.join(HERE, "_ref")
REF_ROOT = os.path.join(REF_DIR, "HairFastGAN")
EXT_DIR = os.path.join(REF_DIR, "ext")


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "hair_swap.py"))


def ref_root() -> str:
    if not available():
        raise RuntimeError(f"reference not staged at {REF_ROOT}: run tools/stage_reference.sh (needs /root/reference)")
    return REF_ROOT


def activate(overlay: bool, skip_fse_reconstruction: bool = False, chdir: bool = True, workdir: str | None = None,
             **install_kwargs) -> str:
    """Put the staged reference (and the stand-ins) on sys.path; returns the reference root.

    workdir: directory holding `pretrained_models/` (see baseline/synth_checkpoints.py).  The reference resolves every
    checkpoint and SEAN's style codes relative to the cwd, so `workdir` gets symlinks to the reference's top-level
    entries and becomes the cwd."""
    root = ref_root()
    os.environ.setdefault("TORCH_EXTENSIONS_DIR", EXT_DIR)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")      # same nvcc line here (no GPU) and on the B200 box
    os.environ.setdefault("MAX_JOBS", "8")
    for p in (STUBS, root, REPO):
        if p in sys.path:
            sys.path.remove(p)
    sys.path[:0] = [root, STUBS, REPO]
    if overlay:
        import hairfastgan_b200.install as hfi
        hfi.install(skip_fse_reconstruction=skip_fse_reconstruction, **install_kwargs)
    if workdir is not None:
        # face_parsing/resnet.py:82-88 fetches torchvision's resnet18 through torch.hub; the synthetic stand-in lives here
        os.environ.setdefault("TORCH_HOME", os.path.join(workdir, "torch_home"))
    if chdir:
        wd = workdir or root
        if workdir is not None:
            os.makedirs(workdir, exist_ok=True)
            for entry in os.listdir(root):
                dst = os.path.join(workdir, entry)
                if entry in ("pretrained_models", "__pycache__") or os.path.lexists(dst):
                    continue
                os.symlink(os.path.join(root, entry), dst)
        os.chdir(wd)
    return root


def cpu_dryrun_patches() -> None:
    """DEBUG ONLY (tools/dryrun_swap_cpu.py, no GPU in the build container): let the stock reference's hard-coded
    'cuda' spots (models/Encoders.py:78,112,143; my_parsing_util.py:81; utils/bicubic.py:45-46; sean_codes) run on the
    CPU so that stubs + synthetic checkpoints can be validated before GPU minutes are spent.  Never used by a test
    that claims parity or by the bench."""
    import torch
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self
    torch.cuda.is_available = lambda: True
    torch.cuda.manual_seed = lambda *a, **k: None
    torch.cuda.manual_seed_all = lambda *a, **k: None

    class _S:
        def synchronize(self):
            return None
    torch.cuda.current_stream = lambda *a, **k: _S()
    torch.cuda.FloatTensor = torch.FloatTensor
    torch.cuda.ByteTensor = torch.ByteTensor
    _device = torch.device

    def _map(d):
        if isinstance(d, str) and d.startswith("cuda"):
            return "cpu"
        if isinstance(d, _device) and d.type == "cuda":
            return _device("cpu")
        return d
    _to = torch.Tensor.to
    torch.Tensor.to = lambda self, *a, **k: _to(self, *[_map(x) for x in a], **{n: _map(v) for n, v in k.items()})
    _mto = torch.nn.Module.to
    torch.nn.Module.to = lambda self, *a, **k: _mto(self, *[_map(x) for x in a], **{n: _map(v) for n, v in k.items()})
    _load = torch.load

    def load(f, map_location=None, **k):
        return _load(f, map_location="cpu", **k)
    torch.load = load
    _type = torch.Tensor.type

    def type_(self, dtype=None, *a, **k):
        if isinstance(dtype, str):
            dtype = dtype.replace("torch.cuda.", "torch.")
        return _type(self, dtype, *a, **k)
    torch.Tensor.type = type_
    for fn in ("randn", "zeros", "ones", "empty", "tensor", "arange", "full", "rand"):
        orig = getattr(torch, fn)

        def wrap(*a, __orig=orig, **k):
            if "device" in k:
                k["device"] = _map(k["device"])
            return __orig(*a, **k)
        setattr(torch, fn, wrap)
    import torch.nn.functional as F
    _interp = F.interpolate

    def interpolate(input, *a, **k):            # CUDA has integer 'nearest'; the CPU kernel does not
        if not input.is_floating_point():
            return _interp(input.double(), *a, **k).to(input.dtype)
        return _interp(input, *a, **k)
    F.interpolate = interpolate
