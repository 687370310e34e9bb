"""`lib.utils.extend_utils.extend_utils` as lib/utils/evaluation_utils.py:16 imports it
(`from lib.utils.extend_utils.extend_utils import uncertainty_pnp, find_nearest_point_idx, uncertainty_pnp_v2`):
the uncertainty-driven PnP and the nearest-neighbour index search, served by pvnet_b200's device code.  The
module's other functions (mesh rasterisation, farthest point sampling) are dataset tooling outside the
inference and evaluation path and are not provided."""
from pvnet_b200.extend_utils import (covariance_to_weights, find_nearest_point_idx, uncertainty_pnp,  # noqa: F401
                                     uncertainty_pnp_batched, uncertainty_pnp_v2)

__all__ = ["uncertainty_pnp", "uncertainty_pnp_batched", "covariance_to_weights", "find_nearest_point_idx",
           "uncertainty_pnp_v2"]
