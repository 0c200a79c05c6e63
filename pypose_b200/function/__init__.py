from .checking import is_lietensor, is_SE3, hasnan
from .linalg import bvv, bmv, bvmv
from .geometry import cart2homo, homo2cart, point2pixel, pixel2point, reprojerr, svdtf, knn
from .spline import chspline, bspline
