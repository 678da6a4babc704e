"""hmse_b200 - the HMSE data-reduction hot path (FastCDC, SHA-256 dedup, preset-dictionary
DEFLATE, MinHash/LSH) as hand-written sm_100a CUDA kernels behind a C ABI (include/hmse.h).

Importing the package does not need a GPU; creating a Context (or calling any API function)
does, and raises if the CUDA library is missing.  The package never imports `oracle`."""
from .config import CDCConfig, SimConfig, gear_table, PAPER_MASK_S, PAPER_MASK_L  # noqa: F401
from ._lib import HmseError, LIB_PATH, load as load_library  # noqa: F401
from .api import Context, default_context, chunk, chunk_files, digest, dedup, compress, compress_bound, inflate, similarity, delta, delta_apply  # noqa: F401
from .ingest import Ingest, IngestStream, ShardedIngest, ShardedSimilarity, IngestResult, HostIngestResult, verify_roundtrip  # noqa: F401,E402
from . import archive, corpus, sharding  # noqa: F401,E402
