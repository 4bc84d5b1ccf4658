"""l-giremi_b200 -- B200-native (sm_100a) implementation of the L-GIREMI
mutual-information step behind the reference's own Python functions.

The directory name carries a hyphen (it mirrors the reference's name), so load
it with ``importlib.import_module("l-giremi_b200")``.

Public surface (same names as the reference where one exists):
    mismatch_pair_mutual_info, mean_mismatch_pair_mutual_info, ecdf   -- drop-ins
    mi_step_batched, mip_and_calls, Batch, Context                     -- batched path
    encode_mismatches, encode_batch, pack_units, PlaneBatch            -- encoder
    partition_lpt, unit_costs, DevicePool, merge_shards, split_means,  -- multi-GPU sharding
    split_means_ipc
    install / uninstall                                                -- patch a loaded `giremi`
"""
from ._lib import (DENSE_DEFAULT, LIB_PATH, MODE_ALL_PAIRS, MODE_COMPACT_OUTPUT, MODE_EMIT_COUNTS, MODE_HET_ONLY, MODE_GRAPH,
                   MODE_SKIP_NONHET, MODE_SPLIT_RECORDS, MODE_TIGHT_INPUT,
                   PAIR_REC, SITE_HET_SNP, SITE_MISMATCH, SITE_SNP, UNIT_DESC, LgmiError)
from .api import (Batch, Context, Pipeline, StepResult, default_device, device_count, ecdf, get_context,
                  mean_mismatch_pair_mutual_info, mi_step_batched, mip_and_calls, mismatch_pair_mutual_info,
                  partition_lpt, site_splice_mutual_info, split_means, split_means_ipc, stream_schedule, stream_steps, unit_costs)
from .encode import (EncodedUnit, PlaneBatch, concat_plane_batches, cs_read_mismatches, encode_batch, encode_mismatches,
                     encode_mismatches_native, pack_units)
from .batched import (analyse_extracted, extract_footprints, extract_region, footprint_bulk_calculation,
                      region_mismatch_analysis)
from .multigpu import DevicePool, MergedResult, merge_shards
from .patch import install, uninstall

__version__ = "0.1.0"
