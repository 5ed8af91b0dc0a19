"""TEST INFRASTRUCTURE ONLY -- loads the *unmodified* reference modules from /root/reference.

The reference package cannot be imported as a package (``import quantized_sae`` dies on the
missing ``baseSAE`` / ``nnba`` modules, see src/quantized_sae/sae/binary.py:7-8), so the
individual source files are executed by path with three import shims:

  * ``baseSAE.SAE``  -> src/quantized_sae/sae/base.py
  * ``nnba.adder``   -> empty module (star-imported, no name is used by any forward)
  * ``SAEs.quantized_matryoshka_SAE`` -> src/quantized_sae/sae/quantized_matryoshka.py

It needs a checkout of the reference project (``QSAE_REFERENCE_ROOT``), which is not part of this
repository. Only the fixture generators ``tests/golden/make_golden*.py`` use it; the product
package, the tests, ``build()``, ``smoke()`` and ``bench.py`` never import this file.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types
from pathlib import Path

REFERENCE_ROOT = Path(os.environ.get("QSAE_REFERENCE_ROOT", "/root/reference"))
_SAE_DIR = REFERENCE_ROOT / "src" / "quantized_sae" / "sae"

_cache: dict[str, types.ModuleType] = {}


def available() -> bool:
    return (_SAE_DIR / "binary.py").is_file()


def _exec(path: Path, name: str) -> types.ModuleType:
    sys.dont_write_bytecode = True  # the reference tree is read-only
    spec = importlib.util.spec_from_file_location(name, str(path))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def load() -> types.SimpleNamespace:
    """Return a namespace with the reference classes (BinarySAE, binary_decoder, ...)."""
    if not available():
        raise FileNotFoundError(f"reference sources not found under {REFERENCE_ROOT}")
    if "ns" in _cache:
        return _cache["ns"]
    base = _exec(_SAE_DIR / "base.py", "baseSAE.SAE")
    pkg = types.ModuleType("baseSAE")
    pkg.SAE = base
    sys.modules["baseSAE"] = pkg
    nnba = types.ModuleType("nnba")
    adder = types.ModuleType("nnba.adder")
    adder.__all__ = []
    nnba.adder = adder
    sys.modules["nnba"] = nnba
    sys.modules["nnba.adder"] = adder
    binary = _exec(_SAE_DIR / "binary.py", "_ref_binary")
    baseline = _exec(_SAE_DIR / "baseline.py", "_ref_baseline")
    ternary = _exec(_SAE_DIR / "ternary.py", "_ref_ternary")
    saes = types.ModuleType("SAEs")
    sys.modules["SAEs"] = saes
    qm = _exec(_SAE_DIR / "quantized_matryoshka.py", "SAEs.quantized_matryoshka_SAE")
    saes.quantized_matryoshka_SAE = qm
    try:
        rq = _exec(_SAE_DIR / "residual_quantized.py", "_ref_residual_quantized")
    except Exception:  # pragma: no cover - optional, not on the hot path
        rq = None
    ns = types.SimpleNamespace(
        SparseAutoencoder=base.SparseAutoencoder,
        binary_decoder=binary.binary_decoder,
        BinarySAE=binary.BinarySAE,
        BaselineSparseAutoencoder=baseline.BaselineSparseAutoencoder,
        STEWeights=ternary.STEWeights,
        TernarySparseAutoencoder=ternary.TernarySparseAutoencoder,
        QuantizedMatryoshkaDecoder=qm.QuantizedMatryoshkaDecoder,
        QuantizedMatryoshkaSAE=qm.QuantizedMatryoshkaSAE,
        ResidualQuantizedSAE=getattr(rq, "ResidualQuantizedSAE", None) if rq else None,
    )
    _cache["ns"] = ns
    _cache["mods"] = dict(binary=binary, baseline=baseline, qm=qm, rq=rq)
    return ns


def load_analysis() -> types.SimpleNamespace:
    """The reference's inference wrapper (src/quantized_sae/inference/framework.py) and analysis script
    (scripts/analysis/dynamic_analysis.py), unmodified. Both import the pre-refactor module names
    (`SAEs.binary_SAE`, `sae_inference_framework`, ...): those are aliased to the shim-loaded modules."""
    ns = load()
    if "analysis" in _cache:
        return _cache["analysis"]
    mods = _cache["mods"]
    saes = sys.modules["SAEs"]
    for alias, mod in (("baseline_SAE", mods["baseline"]), ("binary_SAE", mods["binary"]),
                       ("residual_quantized_matryoshka_SAE", mods["rq"])):
        sys.modules[f"SAEs.{alias}"] = mod
        setattr(saes, alias, mod)
    fw = _exec(REFERENCE_ROOT / "src" / "quantized_sae" / "inference" / "framework.py", "sae_inference_framework")
    da = _exec(REFERENCE_ROOT / "scripts" / "analysis" / "dynamic_analysis.py", "_ref_dynamic_analysis")
    out = types.SimpleNamespace(framework=fw, dynamic_analysis=da, classes=ns)
    _cache["analysis"] = out
    return out
