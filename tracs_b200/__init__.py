"""tracs_b200 -- B200 (sm_100a) implementation of the TRACS pairwise-distance hot path.

Product surface = the C ABI in include/tracs_b200.h (libtracs_b200.so) plus this thin Python
mirror of the reference's `TRACS` extension module. `install_dropin()` makes `import TRACS`
resolve to it, so the reference's tracs/distance.py, tracs/transcluster.py run unchanged."""
import os
import sys

from .api import (pairsnp, trans_dist, lprob_k_given_N, calculate_posteriors, pairsnp_matrix, pairsnp_device, pairsnp_packed,
                  pairsnp_packed_host, pack_nibbles, distance_matrix, distance_matrix_device, write_distance_matrix,
                  min_over_refs, synth_device, int_peak, tc_peak, tc_peak_sustained, last_stats, read_fasta, shard_rowblocks, connected_components, Database,
                  INT32_MAX)

DROPIN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "dropin")


def install_dropin():
    """Puts tracs_b200/dropin (which holds TRACS.py) at the front of sys.path."""
    if DROPIN_DIR not in sys.path:
        sys.path.insert(0, DROPIN_DIR)
    import TRACS  # noqa: F401
    return TRACS
