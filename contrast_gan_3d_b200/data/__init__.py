from .Scaler import FactorZeroCenterScaler, ZeroCenterScaler  # noqa: F401
from .sampler import DevicePatchSampler, pad_amounts, random_crop_lower_bounds  # noqa: F401
from .augment import SpatialTransform2  # noqa: F401
