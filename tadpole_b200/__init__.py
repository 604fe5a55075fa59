"""tadpole_b200 -- B200-native implementation of the TADpole TAD-calling hot path.

Public API mirrors the reference R package (3DGenomes/TADpole, NAMESPACE:3-8):
TADpole(), load_mat(), diffT(), random_bed().  All numeric work runs in
libtadpole_b200.so (hand-written CUDA for sm_100a behind a C ABI, include/tadpole_b200.h).
"""
from .api import TADpole, load_mat, diffT, diffT_batch, diffT_null, random_bed, random_bed_batch, read_matrix, bin_index, Tadpole, LoadedMatrix, SparseCounts, get_context
from ._lib import Context, TadpoleError, assemble
from .hclust import Dendro, find_groups, cutree
from .batch import ContextPool, TADpole_batch, GenomePixels, TADpole_genome, read_bins

__all__ = ["TADpole", "load_mat", "diffT", "diffT_batch", "diffT_null", "random_bed", "random_bed_batch", "read_matrix", "bin_index", "Tadpole", "LoadedMatrix", "SparseCounts",
           "get_context", "ContextPool", "TADpole_batch", "GenomePixels", "TADpole_genome", "read_bins", "Context", "TadpoleError", "assemble", "Dendro", "find_groups", "cutree"]
__version__ = "0.1.0"
