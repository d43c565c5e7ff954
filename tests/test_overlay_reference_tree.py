"""With ``hairfastgan_b200.install.install()`` active, the module structure of the reference files that swap() imports
resolves the hot-path classes to this package.  The structure comes from tests/golden/reference_imports.json
(oracle/gen_golden_imports.py: the reference's own `from X import ...` statements, top-level classes with their method
names and functions, recorded from the original checkout); the test rebuilds a stand-in tree with exactly those names.
Third-party packages the image lacks (dlib, clip, lpips, ...) are replaced by inert stubs; nothing is constructed or
run -- this is about import-time name resolution only.  Runs in a fresh interpreter."""
import json
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_imports.json")

PROBE = textwrap.dedent("""
    import importlib, sys, types
    sys.path.insert(0, %(root)r)
    import hairfastgan_b200.install as hfi
    hfi.install(skip_fse_reconstruction=True)
    sys.path.insert(0, %(ref)r)

    class Stub(types.ModuleType):
        __path__ = []
        def __getattr__(self, name):
            if name.startswith("__"):
                raise AttributeError(name)
            m = Stub(self.__name__ + "." + name); setattr(self, name, m); return m
        def __call__(self, *a, **k):
            return self
        def __iter__(self):
            return iter(())

    for name in ["gdown", "clip", "dlib", "face_alignment", "lpips", "addict", "matplotlib", "matplotlib.pyplot",
                 "cv2", "skimage", "skimage.io", "ranger", "tensorboard_logger", "yaml"]:
        try:
            importlib.import_module(name)
        except Exception:
            sys.modules[name] = Stub(name)

    import models.Net as net, models.Encoders as enc, models.Embedding as emb, models.Blending as blend
    import models.encoder4editing.models.psp as psp
    import models.FeatureStyleEncoder.FSencoder  # noqa: F401  (puts its directory on sys.path, imports `trainer`)
    import models.CtrlHair.external_code.face_parsing.my_parsing_util as parsing
    trainer = sys.modules["trainer"]
    got = {
        "Net.Generator": net.Generator.__module__,
        "Net.FeatureEncoderMult": net.FeatureEncoderMult.__module__,
        "Encoders.FeatureEncoderMult": enc.FeatureEncoderMult.__module__,
        "Encoders.FeatureiResnet": enc.FeatureiResnet.__module__,
        "Encoders.PixelNorm": enc.PixelNorm.__module__,
        "Embedding.BicubicDownSample": emb.BicubicDownSample.__module__,
        "Blending.BicubicDownSample": blend.BicubicDownSample.__module__,
        "Blending.DilateErosion": blend.DilateErosion.__module__,
        "psp.Encoder4Editing": psp.psp_encoders.Encoder4Editing.__module__,
        "trainer.Generator": trainer.Generator.__module__,
        "trainer.fs_encoder_v2": trainer.fs_encoder_v2.__module__,
        "trainer.Trainer.test": "patched" if hasattr(trainer.Trainer.test, "__wrapped__") else "reference",
        "parsing.BiSeNet": parsing.BiSeNet.__module__,
        "parsing.parsing_img": "patched" if hasattr(parsing.FaceParsing_tensor.parsing_img, "__wrapped__") else "reference",
        "Net.Net": net.Net.__module__,
    }
    for k, v in got.items():
        print(k, v)
""")

EXPECTED = {
    "Net.Generator": "hairfastgan_b200.model",
    "Net.FeatureEncoderMult": "hairfastgan_b200.postprocess",
    "Encoders.FeatureEncoderMult": "hairfastgan_b200.postprocess",
    "Encoders.FeatureiResnet": "hairfastgan_b200.postprocess",
    "Encoders.PixelNorm": "hairfastgan_b200.model",
    "Embedding.BicubicDownSample": "hairfastgan_b200.bicubic",
    "Blending.BicubicDownSample": "hairfastgan_b200.bicubic",
    "Blending.DilateErosion": "hairfastgan_b200.masks",
    "psp.Encoder4Editing": "hairfastgan_b200.encoders",
    "trainer.Generator": "hairfastgan_b200.fse_model",
    "trainer.fs_encoder_v2": "hairfastgan_b200.encoders",
    "trainer.Trainer.test": "patched",
    "parsing.BiSeNet": "hairfastgan_b200.bisenet",
    "parsing.parsing_img": "patched",
    "Net.Net": "models.Net",                      # the orchestration class stays the reference's
}


def _stand_in_tree(dst):
    """One file per recorded module: its import statements (an import this environment cannot satisfy is left out, as
    the stubs below do for third-party packages), then its functions and classes as empty bodies."""
    spec = json.load(open(GOLDEN))
    packages = set()
    for rel, d in spec.items():
        parts = rel[:-3].split("/")
        packages.update("/".join(parts[:i]) for i in range(1, len(parts)))
        for mod, _ in d["imports"]:
            if mod.split(".")[0] in ("models", "utils"):
                mp = mod.split(".")
                packages.update("/".join(mp[:i]) for i in range(1, len(mp) + 1))
    packages -= {rel[:-3] for rel in spec}
    for pkg in packages:
        os.makedirs(os.path.join(dst, pkg), exist_ok=True)
        open(os.path.join(dst, pkg, "__init__.py"), "a").close()
    for rel, d in spec.items():
        lines = ["import os", "import sys"]
        if d["sys_path_insert_own_dir"]:
            lines.append("sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))")
        for mod, names in d["imports"]:
            lines += ["try:", f"    from {mod} import {', '.join(names)}", "except ImportError:", "    pass"]
        lines += [f"def {fn}(*args, **kwargs):\n    pass" for fn in d["functions"]]
        for cls, methods in d["classes"].items():
            lines.append(f"class {cls}:")
            lines += [f"    def {m}(self, *args, **kwargs):\n        pass" for m in methods] or ["    pass"]
        with open(os.path.join(dst, rel), "w") as f:
            f.write("\n".join(lines) + "\n")


def test_reference_imports_resolve_to_this_package(tmp_path):
    ref = tmp_path / "reference"
    _stand_in_tree(str(ref))
    p = subprocess.run([sys.executable, "-c", PROBE % {"root": ROOT, "ref": str(ref)}], capture_output=True, text=True,
                       timeout=600, cwd=str(tmp_path))
    assert p.returncode == 0, p.stderr[-3000:]
    got = dict(line.split(" ", 1) for line in p.stdout.strip().splitlines() if " " in line)
    assert got == EXPECTED, {k: (got.get(k), v) for k, v in EXPECTED.items() if got.get(k) != v}
