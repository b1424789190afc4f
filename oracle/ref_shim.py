"""Import-time stubs that let the UNMODIFIED reference (``/root/reference``) be imported
in this container.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

The reference needs ``timm``, ``yacs``, ``omegaconf``, ``matplotlib``, ``equilib`` and
``imageio`` at import time (SURVEY.md section 8c); none of them does inference arithmetic:

* ``timm.models.layers.DropPath``  -> identity in eval mode (mix_transformers.py:11, convnext.py:13)
* ``timm.models.layers.to_2tuple`` / ``trunc_normal_`` -> trivial / ``torch.nn.init.trunc_normal_``
* ``yacs.config.CfgNode``          -> attribute dict with ``merge_from_file`` (PyYAML) and ``freeze``
  (config/config.py:1, perspectivefields.py:124-131)
* ``omegaconf.DictConfig``         -> empty class (utils/config.py:7)
* ``matplotlib*``, ``equilib`` (``__version__ == "0.3.0"`` is asserted in utils/panocam.py:8),
  ``imageio``                      -> empty modules

Nothing here is imported by the product package or by the tests: only the golden generators
(tests/golden/make_golden*.py) call ``load_reference``, and the tests compare with what they stored.
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("PF_REFERENCE_ROOT", "/root/reference")


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "perspective2d"))


def _module(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def _install_stubs():
    import torch
    import yaml

    if "timm" not in sys.modules:

        class DropPath(torch.nn.Module):
            def __init__(self, drop_prob=0.0, *a, **k):
                super().__init__()
                self.drop_prob = drop_prob

            def forward(self, x):
                assert not self.training, "stub DropPath is eval-only"
                return x

        def to_2tuple(x):
            return tuple(x) if isinstance(x, (tuple, list)) else (x, x)

        layers = _module(
            "timm.models.layers",
            DropPath=DropPath,
            to_2tuple=to_2tuple,
            trunc_normal_=torch.nn.init.trunc_normal_,
        )
        models = _module("timm.models", layers=layers)
        _module("timm", models=models)

    if "yacs" not in sys.modules:

        class CfgNode(dict):
            def __getattr__(self, k):
                try:
                    return self[k]
                except KeyError as e:
                    raise AttributeError(k) from e

            def __setattr__(self, k, v):
                self[k] = v

            def _merge(self, other):
                for k, v in other.items():
                    if isinstance(v, dict):
                        node = self.get(k)
                        if not isinstance(node, CfgNode):
                            node = CfgNode()
                            self[k] = node
                        node._merge(v)
                    else:
                        self[k] = v

            def merge_from_file(self, path):
                with open(path) as f:
                    self._merge(yaml.safe_load(f))

            def freeze(self):
                pass

            def clone(self):
                import copy

                return copy.deepcopy(self)

        config = _module("yacs.config", CfgNode=CfgNode)
        _module("yacs", config=config)

    if "omegaconf" not in sys.modules:
        _module("omegaconf", DictConfig=type("DictConfig", (), {}))

    if "matplotlib" not in sys.modules:
        mpl = _module("matplotlib")
        mpl.pyplot = _module("matplotlib.pyplot")
        mpl.colors = _module("matplotlib.colors")
        mpl.figure = _module("matplotlib.figure")
        mpl.cm = _module("matplotlib.cm")
        mpl.backends = _module("matplotlib.backends")
        mpl.backends.backend_agg = _module(
            "matplotlib.backends.backend_agg", FigureCanvasAgg=type("FigureCanvasAgg", (), {})
        )

    if "equilib" not in sys.modules:
        _module("equilib", __version__="0.3.0", equi2pers=None, grid_sample=None)
    if "imageio" not in sys.modules:
        _module("imageio")
    if "albumentations" not in sys.modules:
        _module("albumentations")


def load_reference():
    """Return the reference's ``perspective2d`` package (imported unmodified)."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    _install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import perspective2d  # noqa: E402

    if not os.path.realpath(perspective2d.__file__).startswith(os.path.realpath(REFERENCE_ROOT)):
        raise RuntimeError("a different 'perspective2d' shadows the reference: " + perspective2d.__file__)
    return perspective2d
