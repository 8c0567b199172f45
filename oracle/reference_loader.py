"""Load the UNMODIFIED reference model files from a checkout of the original project.

TEST INFRASTRUCTURE ONLY.  The checkout is not part of this repository: it is looked for in
``oracle/_ref`` (git-ignored) or where ``SN_REFERENCE_ROOT`` points, and without it ``available()``
is False.  Used by oracle/make_golden*.py (fixture generation) and by the live-reference tests
(skipped when the checkout is absent; tests/golden/ holds what the original computed).

One source-text shim is applied at load time (SURVEY.md section 8c):
``top_k_words / self.vocab_size`` -> ``//`` so that ``sample()`` indexes with integers on
torch >= 1.5 (stylenet/model.py:249, model_att.py:381, nic/model.py:162,
nic/model_att.py:261, app/backend/model.py:170,442).  Nothing else is changed.
"""
import importlib.util
import os
import sys
import types

REF_ROOT = os.environ.get("SN_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")

_FILES = {
    "stylenet": "stylenet/model.py",
    "stylenet_att": "stylenet/model_att.py",
    "nic": "nic/model.py",
    "nic_att": "nic/model_att.py",
    "app": "app/backend/model.py",
    "app_att": "app/backend/model_att.py",
    "stylenet_utils": "stylenet/utils.py",
    "seq2seq": "seq2seq/model.py",
}
_cache = {}


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, _FILES["stylenet"]))


def load(name: str) -> types.ModuleType:
    """Return the reference module ``name`` (one of _FILES) with the ``//`` shim."""
    if name in _cache:
        return _cache[name]
    path = os.path.join(REF_ROOT, _FILES[name])
    with open(path, "r") as fh:
        src = fh.read()
    src = src.replace("top_k_words / self.vocab_size", "top_k_words // self.vocab_size")
    mod = types.ModuleType("sn_reference_" + name)
    mod.__file__ = path
    exec(compile(src, path, "exec"), mod.__dict__)
    _cache[name] = mod
    return mod
