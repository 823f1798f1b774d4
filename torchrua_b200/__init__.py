"""torchrua_b200 -- a B200-native (sm_100a) implementation of TorchRua's ragged-sequence hot path behind
TorchRua's own Python API.  ``import torchrua_b200 as torchrua`` is the intended drop-in.

Same façade as the reference (torchrua/__init__.py:1-8): every public name of every submodule is
re-exported.  Like the reference, importing this package patches ``torch.Tensor.__getitem__`` /
``__setitem__`` and adds the ragged-sequence methods to ``torch.nn.utils.rnn.PackedSequence``.
"""
from torchrua_b200.utils import *  # noqa: F401,F403
from torchrua_b200.layout import *  # noqa: F401,F403
from torchrua_b200.core import *  # noqa: F401,F403
from torchrua_b200.compose import *  # noqa: F401,F403
from torchrua_b200.conv import *  # noqa: F401,F403
from torchrua_b200.crf import *  # noqa: F401,F403
from torchrua_b200.delta import *  # noqa: F401,F403
from torchrua_b200.detach import *  # noqa: F401,F403
from torchrua_b200.mask import *  # noqa: F401,F403
from torchrua_b200.reduce import *  # noqa: F401,F403
from torchrua_b200.scan import *  # noqa: F401,F403
from torchrua_b200.segment import *  # noqa: F401,F403
from torchrua_b200.ssm import *  # noqa: F401,F403
from torchrua_b200.ssd import *  # noqa: F401,F403
from torchrua_b200.select import *  # noqa: F401,F403

__version__ = '0.1.0'
