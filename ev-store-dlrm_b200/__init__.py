"""evstore-b200: B200-native embedding-lookup hot path of EVStore (EvLFU cache C1, mixed-precision
tiers C2, approximate embeddings C3) behind the reference's cache_manager / storage_manager /
apply_emb_evstore surface.  The directory name has a hyphen: import it with
``importlib.import_module("ev-store-dlrm_b200")`` (``__graft_entry__`` does)."""
from ._native import EvsError, load_library, LIB_PATH, SYMBOLS  # noqa: F401
from .cache_manager import CacheConfig, EvStore, host_rows, state_info, to_host_rows  # noqa: F401
from . import altkeys, codecs, cpp_socket_client, dlrm_ops, evstore_utils, sharded, storage_manager, workload  # noqa: F401
