"""allwave_b200 -- B200-native (sm_100a) batched bidirectional wavefront aligner behind
allwave's alignment path.  The compute lives in liballwave_cuda.so (C ABI, include/allwave_cuda.h);
this package is the host-side mirror of the reference interface used by tests and bench.py."""
from . import _cabi  # noqa: F401
from ._cabi import (  # noqa: F401
    AW_EALIGN, AW_ECALLBACK, AW_ECUDA, AW_EINVAL, AW_ENODEVICE, AW_ENOMEM, AW_EUNSUPPORTED, AW_EWORKSPACE,
    AW_FLAG_CIGAR_BYTES, AW_FLAG_CS, AW_FLAG_CS_LONG, AW_FLAG_NO_PAF, AW_FLAG_ORDERED, AW_FLAG_PAF_BLOCKS, AW_FLAG_SCORE_ONLY, AW_OK, AW_ORIENT_FORWARD, AW_ORIENT_MASH,
    AW_ORIENT_WFA, AW_SCOPE_ALIGNMENT, AW_SCOPE_SCORE,
    Aligner, AllwaveError, Batch, Context, build, make_params,
)
