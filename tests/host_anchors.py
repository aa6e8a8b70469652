"""libcpecan.so's host anchorer (host/anchors.c) through ctypes: getBlastPairsForPairwiseAlignmentParameters, the reference that the
device anchors of cpb_batch_create_anchored are held to.  Calls release the GIL, so host threads can anchor pairs side by side."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "cpecan_b200", "lib", "libcpecan.so")


class HostParams(C.Structure):
    """PairwiseAlignmentParameters (include/cpecan/pairwiseAligner.h)"""

    _fields_ = [("threshold", C.c_double), ("minDiagsBetweenTraceBack", C.c_int64), ("traceBackDiagonals", C.c_int64),
                ("diagonalExpansion", C.c_int64), ("constraintDiagonalTrim", C.c_int64), ("anchorMatrixBiggerThanThis", C.c_int64),
                ("repeatMaskMatrixBiggerThanThis", C.c_int64), ("splitMatrixBiggerThanThis", C.c_int64),
                ("alignAmbiguityCharacters", C.c_bool), ("gapGamma", C.c_float), ("dynamicAnchorExpansion", C.c_bool)]


class _StList(C.Structure):
    """the head of host/containers.c's stList: its item array and length"""

    _fields_ = [("items", C.POINTER(C.c_void_p)), ("length", C.c_int64)]


class HostAnchorer:
    def __init__(self, path=LIB):
        L = C.CDLL(path)
        L.getBlastPairsForPairwiseAlignmentParameters.restype = C.c_void_p
        L.getBlastPairsForPairwiseAlignmentParameters.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int64, C.POINTER(HostParams)]
        L.stIntTuple_get.restype = C.c_int64
        L.stIntTuple_get.argtypes = [C.c_void_p, C.c_int64]
        L.stList_destruct.argtypes = [C.c_void_p]
        self.L = L

    @staticmethod
    def params(p):
        """HostParams with the fields of a cpecan_b200.CpbParams"""
        h = HostParams()
        for name, _ in HostParams._fields_:
            setattr(h, name, getattr(p, name))
        return h

    def blast_pairs(self, sx, sy, hp):
        """the stList handle of one pair's anchors (free with read)"""
        return self.L.getBlastPairsForPairwiseAlignmentParameters(sx, sy, len(sx), len(sy), C.byref(hp))

    def read(self, handle):
        """-> int64 [m, 3] (x, y, expansion); frees the list"""
        head = C.cast(handle, C.POINTER(_StList)).contents
        m = head.length
        out = np.zeros((m, 3), dtype=np.int64)
        if m:
            items = np.ctypeslib.as_array(C.cast(head.items, C.POINTER(C.c_uint64)), shape=(m,))
            if m == 1 or np.all(np.diff(items.astype(np.int64)) == 32):
                # cpecan_tripleList_construct cuts the tuples from one slab: (length word, x, y, expansion) every 32 bytes
                out[:] = np.ctypeslib.as_array((C.c_int64 * (4 * m)).from_address(int(items[0]))).reshape(m, 4)[:, 1:]
            else:
                for i in range(m):
                    out[i] = [self.L.stIntTuple_get(C.c_void_p(int(items[i])), k) for k in range(3)]
        self.L.stList_destruct(handle)
        return out

    def anchors(self, sx, sy, hp):
        return self.read(self.blast_pairs(sx, sy, hp))
