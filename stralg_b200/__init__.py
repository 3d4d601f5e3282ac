"""stralg_b200 -- B200-native suffix array / BWT / FM-index engine behind stralg's hot-path API.

The package holds only what the hot path needs: ``csrc/`` (sm_100a CUDA kernels + the C ABI of
``include/b200sa.h``) and this thin host-side mirror of the reference's interface.  There is no
CPU fallback: everything calls into ``lib/libb200sa.so``.
"""
from ._lib import B200saError, LIB_PATH, load  # noqa: F401
from .index import (RecordsRemap, RemapTable, SuffixArrayIndex, build_complete_table, pack_reads, qsort_sa_construction,  # noqa: F401
                    search_sharded_packed,
                    sa_is_construction, sa_is_mem_construction, skew_sa_construction)
