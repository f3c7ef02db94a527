"""outerspace_b200 -- B200-native outer-product SpGEMM engine.

Drop-in for the functional multiply/merge path of anneouyang/OuterSPACE (TaskProvider in
simulator/SimOuterSPACE.cpp, loaders in simulator/SimSpGEMM.cpp).  The compute lives in
``libosp_b200.so`` (hand-written sm_100a CUDA behind the C ABI of include/osp_b200.h);
this package is the thin host mirror of the reference's interface.
"""
from .formats import COO, CSRMatrix, ELEM  # noqa: F401
from .api import (  # noqa: F401
    DeviceCOO, DuplicateEntry, Engine, OspError, Result, TaskProvider, coo2csr, csc2rawcompact, csr2compact, default_engine, load_library,
    readcoo,
)
