"""Python copy of the launch plan of segscan_kernel (torchrua_b200/csrc/scan.cu: with_scan_op + make_plan).

test_scan_plan.py pins it on the CPU against the workspace size the library reports; test_gpu_scan_backward.py uses it
to name the regime (vector width, threads across a row, column blocks, rows per chunk) each case runs in and to bound
the depth of the combination tree a result went through."""
from collections import namedtuple

import torch

THREADS = 256   # kScanThreads
MAX_TPC = 32    # kMaxTPC

# rows per thread group (Op::kRG) of each operator kind
KRG = {'sum': 16, 'lse': 16, 'ext': 8, 'lse_bwd': 4, 'run_bwd': 8, 'linrec': 6, 'linrec_bwd': 8}
# the kernel's C++ operator of each kind
OP_NAME = {'sum': 'OpSum', 'lse': 'OpLse', 'lse_bwd': 'OpLseBwd', 'run_bwd': 'OpRunBwd', 'linrec': 'OpLinRec',
           'linrec_bwd': 'OpLinRecBwd'}
# (element bytes, accumulator bytes, C++ type) per payload dtype
DTYPE = {torch.float32: (4, 4, 'float'), torch.float64: (8, 8, 'double'), torch.float16: (2, 4, '__half'),
         torch.bfloat16: (2, 4, '__nv_bfloat16')}
# scan op -> (forward kind, backward kind); cumsum's gradient is the sum scan run the other way
SCAN_KINDS = {'sum': ('sum', 'sum'), 'logsumexp': ('lse', 'lse_bwd'), 'max': ('ext', 'run_bwd'),
              'min': ('ext', 'run_bwd')}

Plan = namedtuple('Plan', 'V tpc G R ncb chunks total smem')


def _cdiv(a, b):
    return -(-a // b)


def vec_width(dtype):
    """elements per 16-byte vector"""
    return 16 // DTYPE[dtype][0]


def state_bytes(kind, dtype):
    """sizeof(Op::S): the accumulator for sum / logsumexp, a pair for the others ((value, int32 index) of max / min is
    padded to the accumulator's alignment)"""
    acc = DTYPE[dtype][1]
    return acc if kind in ('sum', 'lse') else 2 * acc


def plan(kind, rows, H, dtype, aligned=True):
    """the plan make_plan<Op> builds for `kind` over `rows` positions of H columns; aligned: every pointer of the call is
    16-byte aligned (with_scan_op falls back to one element per thread otherwise, and when H is not a multiple of the
    vector)"""
    VV = vec_width(dtype)
    V = VV if aligned and H % VV == 0 else 1
    vecs = _cdiv(H, V)
    tpc = 1
    while tpc < MAX_TPC and tpc < vecs:
        tpc <<= 1
    G = THREADS // tpc
    R = G * KRG[kind]
    ncb = _cdiv(vecs, tpc)
    chunks = _cdiv(rows, R)
    sb = state_bytes(kind, dtype)
    flag_bytes = _cdiv(16 + 4 * chunks * ncb, 256) * 256
    total = flag_bytes + 2 * chunks * ncb * tpc * V * sb
    # dynamic shared memory of launch_op: row, position (and sequence for the linear recurrence) per row, the decode
    # flags, THREADS x V states and THREADS start flags
    per_row = 25 if kind in ('linrec', 'linrec_bwd') else 17
    smem = R * per_row + sb * THREADS * V + 4 * THREADS
    return Plan(V, tpc, G, R, ncb, chunks, total, smem)


def workspace_bytes(kind, rows, H, dtype):
    """the workspace the library asks for: the larger plan of the two widths the kernel may run at"""
    if rows == 0 or H == 0:
        return 0
    return max(plan(kind, rows, H, dtype, aligned).total for aligned in (True, False))


def instance(kind, dtype, V, op=None):
    """the kernel instance name as the profiler shows it, namespaces and spaces removed"""
    t = DTYPE[dtype][2]
    if kind == 'ext':
        return f'segscan_kernel<OpExt<{t},{V},{str(op == "max").lower()}>>'
    return f'segscan_kernel<{OP_NAME[kind]}<{t},{V}>>'
