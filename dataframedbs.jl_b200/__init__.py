"""dfdb_b200 -- B200-native column-scan path of DataFrameDBs.jl behind the reference's own API.

Host side mirrors the reference's Julia API for this path (open_table / DFTable / DFView / DFColumn,
`table[predicate, cols]`, materialize, nrow and the aggregate reductions); every scan is executed by
hand-written sm_100a CUDA kernels in `lib/libdfdb_b200.so` through the C ABI of include/dfdb_b200.h.
There is no CPU fallback: using a scan without the built CUDA library raises.
"""
from .plan import (ArgumentError, BlockBroadcasting, ColRef, InSet, JRange, JType, Projection, R,  # noqa: F401
                   SelectionQueue, add, encode_plan, required_columns)
from .api import (DFColumn, DFTable, DFView, FlatStringsVector, Frame, coalesce, count, endswith, head, isin,  # noqa: F401
                  ismissing, materialize, maximum, mean, minimum, ncol, nrow, open_table, projection, selection, selproj,
                  startswith, sum, aggregate, create_table, groupreduce, aggregate_all, nrow_all, pruned_blocks, fold, agg_sum, agg_min, agg_max, plan_bytes, selection_mask, selection_indices, size,
                  issameselection, issametable, view_from_columns, resolve_sharded_selection, unique, unique_all, unique_merge,
                  groupreduce_all, groupreduce_local, groupreduce_merge)
from . import _capi  # noqa: F401
from ._capi import DfdbError, LOAD_DECODED, LOAD_HBM, LOAD_HOST  # noqa: F401
