"""latok_b200 -- LaTok's tokenization hot path (characters -> feature bits -> split mask -> token
spans -> per-token feature sums) as hand-written sm_100a CUDA behind LaTok's own Python API.

    from latok_b200.core.default_tokenizer import tokenize, featurize, tokenize_batch
    import latok_b200; latok_b200.install_as_latok()   # `import latok.core.default_tokenizer` now resolves here
    from latok_b200.vocab import Vocab     # token counts and integer token ids on the GPU (Counter / dict lookup)

Everything numeric happens in liblatok_b200.so (C ABI: include/latok_b200.h).  There is no CPU
fallback: without the library or without a CUDA device the compute calls raise.
"""
import sys as _sys

__version__ = "0.1.0"


def install_as_latok():
    """Register this package under the reference's module names (latok, latok.latok, latok.core,
    latok.core.offsets / latok_utils / default_tokenizer) so existing imports keep working."""
    import importlib
    import types
    if "latok" in _sys.modules and not getattr(_sys.modules["latok"], "__latok_b200__", False):
        raise ImportError("a different 'latok' package is already imported")
    ext = importlib.import_module(".latok", __name__)
    core = importlib.import_module(".core", __name__)
    mods = {name: importlib.import_module(".core." + name, __name__)
            for name in ("offsets", "latok_utils", "default_tokenizer")}
    top = types.ModuleType("latok")
    top.__latok_b200__ = True
    top.__path__ = []
    top.__version__ = __version__
    top.latok = ext
    top.core = core
    _sys.modules["latok"] = top
    _sys.modules["latok.latok"] = ext
    _sys.modules["latok.core"] = core
    for name, mod in mods.items():
        _sys.modules["latok.core." + name] = mod
    return top
