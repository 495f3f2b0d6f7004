"""zstdlite_b200: B200-native Zstandard codec behind zstdlite's API (see DESIGN.md)."""
from .api import (ZstdError, zstd_cctx, zstd_dctx, zstd_compress, zstd_decompress, zstd_serialize, zstd_unserialize, zstd_info, zstd_dict_id, zstd_train_dict_compress, zstd_train_dict_serialize,
                  zstd_version, zstd_compress_stream, zstd_decompress_stream, decompress_batch, compress_batch, BatchPlan, is_error, error_name,
                  zstd_seek_table, zstd_decompress_range, zstd_decompress_ranges, zstd_frames)  # noqa: F401
