"""cpecan_b200 -- Python driver (ctypes) over libcpecan_b200.so, the B200-native pair-HMM engine.

The product is the C-ABI shared library (include/cpecan_b200.h, built from cpecan_b200/csrc by
``__graft_entry__.build()`` / ``make -f cpecan_b200/csrc/Makefile``).  This package only binds it for the
tests and bench.py; function names mirror cPecan's C API (inc/pairwiseAligner.h, inc/stateMachine.h).
There is no fallback: importing the package without the built library raises.
"""
from .binding import (  # noqa: F401
    LIB_PATH,
    CpbError,
    CpbModel,
    CpbParams,
    CpbRunStats,
    Context,
    Batch,
    MODE_ALIGNED_PAIRS,
    MODE_ALIGNED_PAIRS_INDELS,
    MODE_EXPECTATIONS,
    MODE_FORWARD,
    SCORE_IDENTITY,
    SCORE_IDENTITY_IGNORING_GAPS,
    SCORE_POSTERIOR,
    SCORE_POSTERIOR_IGNORING_GAPS,
    fiveState,
    fiveStateAsymmetric,
    threeState,
    threeStateAsymmetric,
    PAIR_ALIGNMENT_PROB_1,
    hmm_len,
    lib,
    pairwiseAlignmentBandingParameters_construct,
    stateMachine5_construct,
    stateMachine3_construct,
    hmm_getStateMachine,
    getSplitPoints,
    default_context,
    getAlignedPairs,
    getAlignedPairsWithIndels,
    getExpectations,
    getAlignedPairsUsingAnchors,
    getAlignedPairsWithIndelsUsingAnchors,
    getExpectationsUsingAnchors,
    computeForwardProbability,
    getShiftedMEAAlignment,
)
