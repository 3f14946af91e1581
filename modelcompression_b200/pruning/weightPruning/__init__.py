from .layers import MaskedConv2d, MaskedLinear  # noqa: F401
from .methods import filter_prune, prune_one_filter, quick_filter_prune, weight_prune  # noqa: F401
from .utils import are_masks_consistent, arg_nonzero_min, prune_rate, to_var  # noqa: F401
