"""Shared helpers for tests/, bench.py and __graft_entry__.py: package import (the package directory is
literally `vit.cpp_b200`, which is not an importable identifier) and cached synthetic model files."""
import importlib.util
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_DIR = os.path.join(ROOT, "vit.cpp_b200")
# generated model files live outside the tree (which may be read-only) and are shared by later runs of the same user
CACHE = os.environ.get("VITB200_CACHE", os.path.join(tempfile.gettempdir(), f"vitb200-cache-{os.getuid()}"))


def load_pkg():
    """import the package in `vit.cpp_b200/` under the module name `vit_cpp_b200`."""
    if "vit_cpp_b200" in sys.modules:
        return sys.modules["vit_cpp_b200"]
    spec = importlib.util.spec_from_file_location(
        "vit_cpp_b200", os.path.join(PKG_DIR, "__init__.py"), submodule_search_locations=[PKG_DIR])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["vit_cpp_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


pkg = load_pkg()
gf = pkg.ggml_file


def model_path(config: str, ftype: str = "f16", seed: int = 0) -> str:
    """Path of a cached synthetic model file.  q8_0 files come from the package's own restatement of the reference's quantize.cpp
    (vit.cpp_b200/convert.py, byte-identical to the reference binary: tests/test_oracle.py); the other block formats from the
    reference's quantize binary (oracle/_ref/quantize) applied to the f16 file."""
    os.makedirs(CACHE, exist_ok=True)
    path = os.path.join(CACHE, f"vit-{config}-{ftype}-s{seed}.gguf")
    if os.path.exists(path):
        return path
    tmp = path + f".tmp{os.getpid()}"
    if ftype in ("f16", "f32"):
        gf.write_synthetic(tmp, config, 1 if ftype == "f16" else 0, seed=seed)
    elif ftype == "bf16w":  # bf16-rounded weights stored as f32 (SURVEY.md 8c, bf16 config oracle)
        gf.write_synthetic(tmp, config, 0, seed=seed, round_bf16=True)
    elif ftype == "q8_0":
        pkg.convert.quantize_model_file(model_path(config, "f16", seed), tmp, "q8_0")
    elif ftype in gf.QUANT_NAMES:
        from oracle import ref
        subprocess.check_call([ref.QUANTIZE_BIN, model_path(config, "f16", seed), tmp, str(gf.QUANT_NAMES[ftype])],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    else:
        raise ValueError(ftype)
    os.replace(tmp, path)
    return path
