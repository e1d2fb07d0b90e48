"""Import the UNMODIFIED reference (lucidrains/DALLE-pytorch) from its build under oracle/_ref (oracle/build_ref.py, run by
`__graft_entry__.build()`), else from the reference checkout itself.

TEST / MEASUREMENT INFRASTRUCTURE ONLY -- never imported by the product package.  Users: oracle/make_golden.py (generates
the committed fixtures under tests/golden/), the tests that patch the reference's own classes (`patch_dalle_pytorch()`
rebinding, the drop-in GPU test, GraphedDecoder driving a patched reference model), and bench.py's reference legs
(`--impl reference`, `cpu_baseline`, `gpu_eager_baseline`), which time the reference's own `DALLE(...)` stock code path.

Mechanism (SURVEY.md §8(c)): register a synthetic package object `dalle_pytorch` whose __path__ points
at <root>/dalle_pytorch so that its __init__.py (which pulls tokenizers / vae deps that are not
installed) is skipped, and put oracle/shims (restated rotary_embedding_torch, stubs for
axial_positional_embedding / omegaconf / taming) on sys.path.
"""
import importlib
import os
import sys
import types

_HERE = os.path.dirname(os.path.abspath(__file__))
_SHIMS = os.path.join(_HERE, 'shims')
BUILD_ROOT = os.path.join(_HERE, '_ref')                  # written by oracle/build_ref.py, git-ignored
DEFAULT_SOURCE = '/root/reference'                        # default location of the reference checkout; $DALLE_REFERENCE_ROOT overrides


def is_reference_root(path):
    return bool(path) and os.path.isfile(os.path.join(path, 'dalle_pytorch', 'dalle_pytorch.py'))


def source_root():
    """The reference checkout to build oracle/_ref from, or None where none is readable."""
    for c in (os.environ.get('DALLE_REFERENCE_ROOT'), DEFAULT_SOURCE):
        if is_reference_root(c):
            return c
    return None


REF_ROOT = None


def resolve():
    """Sets REF_ROOT to the copy under oracle/_ref if there is one, else to the checkout; returns it, or None when neither exists.
    oracle/build_ref.py calls it again after (re)building the copy."""
    global REF_ROOT
    REF_ROOT = next((c for c in (BUILD_ROOT, source_root()) if is_reference_root(c)), None)
    return REF_ROOT


resolve()


def reference_available():
    return is_reference_root(REF_ROOT)


def import_reference():
    """Returns a namespace with the reference's DALLE, DiscreteVAE, Transformer, Attention, ... classes."""
    if not reference_available():
        raise RuntimeError(f'reference not found in {BUILD_ROOT} (run oracle/build_ref.py next to a reference checkout)')
    if _SHIMS not in sys.path:
        sys.path.insert(0, _SHIMS)
    if 'dalle_pytorch' not in sys.modules or not getattr(sys.modules['dalle_pytorch'], '_is_ref_shim', False):
        pkg = types.ModuleType('dalle_pytorch')
        pkg.__path__ = [os.path.join(REF_ROOT, 'dalle_pytorch')]
        pkg._is_ref_shim = True
        sys.modules['dalle_pytorch'] = pkg
    ns = types.SimpleNamespace()
    ns.attention = importlib.import_module('dalle_pytorch.attention')
    ns.transformer = importlib.import_module('dalle_pytorch.transformer')
    ns.reversible = importlib.import_module('dalle_pytorch.reversible')
    ns.dalle = importlib.import_module('dalle_pytorch.dalle_pytorch')
    ns.DALLE = ns.dalle.DALLE
    ns.DiscreteVAE = ns.dalle.DiscreteVAE
    ns.Transformer = ns.transformer.Transformer
    ns.Attention = ns.attention.Attention
    ns.SparseAxialCausalAttention = ns.attention.SparseAxialCausalAttention
    ns.SparseConvCausalAttention = ns.attention.SparseConvCausalAttention
    return ns
