from .reproj import PoseReproj, TwoPoseReproj
from .pgo import PoseGraph
from .ba import BundleAdjustment
from .imu_preintegrator import IMUPreintegrator
from .loss import GeodesicLoss, geodesic_loss
from .pnp import EPnP
from .icp import ICP
