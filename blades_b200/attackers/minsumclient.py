"""Min-Sum attacker (Shejwalkar & Houmansadr, NDSS 2021): every Min-Sum client uploads ``mu - g * p``, with ``g`` the
largest scale whose summed squared distance to the honest updates stays within that of the most outlying honest
update (``sum_i ||m - u_i||^2 <= max_i sum_j ||u_i - u_j||^2``).  Needs no knowledge of the aggregator.

Fused like ``MinmaxClient`` (virtual rows, Gram pass over ``[U; q]``, scale search on the device); the callback is
the unfused path.  See ``_agr`` for the shared math."""
from ._agr import ScaledDeviationClient

__all__ = ["MinsumClient"]


class MinsumClient(ScaledDeviationClient):
    kind = "minsum"
