"""Drop-in alias: ``import torchrua`` resolves to the B200-native implementation in ``torchrua_b200`` --
same public names, same module tree (``torchrua.reduce``, ``torchrua.layout.cat``, ``torchrua.select.roll`` ...).
Nothing is implemented here."""
import importlib
import sys

import torchrua_b200 as _impl
from torchrua_b200 import *  # noqa: F401,F403

__version__ = _impl.__version__

for _name in ('utils', 'layout', 'layout.cat', 'layout.left', 'layout.right', 'layout.pack', 'core', 'core.cast',
              'core.get', 'core.set', 'core.view', 'conv', 'crf', 'delta', 'mask', 'reduce', 'scan', 'segment', 'ssm',
              'ssd', 'select', 'select.head', 'select.last', 'select.rev', 'select.roll', 'select.trunc', 'detach', 'compose',
              'shard'):
    sys.modules[f'{__name__}.{_name}'] = importlib.import_module(f'torchrua_b200.{_name}')
for _name in ('utils', 'layout', 'core', 'reduce', 'segment', 'select', 'detach', 'shard'):
    globals()[_name] = sys.modules[f'{__name__}.{_name}']
# like the reference, the star imports leave ``torchrua.mask`` and ``torchrua.compose`` bound to the FUNCTIONS
# of those names (torchrua/__init__.py:1-8); the modules stay reachable through sys.modules / ``import torchrua.mask``
mask = _impl.mask
compose = _impl.compose
