"""Min-Max attacker (Shejwalkar & Houmansadr, NDSS 2021): every Min-Max client uploads ``mu - g * p``, with ``g`` the
largest scale whose malicious update is no farther from any honest update than the two farthest honest updates are
from each other (``max_i ||m - u_i||^2 <= max_{i,j} ||u_i - u_j||^2``).  Needs no knowledge of the aggregator.

B200 path: ``fused_spec()`` describes the attack as virtual rows.  The deviation ``p`` and the distances come from
one Gram pass over ``[U; q]``, the scale search runs on the device (csrc/cuda/gram_solve.cu) and the aggregation
kernels read the resulting parameter from device memory -- no host sync, so the round stays one CUDA graph.  The
callback below is the unfused path (custom aggregators, ``fuse_attack=False``); see ``_agr`` for the shared math."""
from ._agr import ScaledDeviationClient

__all__ = ["MinmaxClient"]


class MinmaxClient(ScaledDeviationClient):
    kind = "minmax"
