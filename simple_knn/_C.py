"""simple-knn's native module: distCUDA2(points [P, 3] float32 CUDA) -> [P], the mean squared distance to the 3 nearest
other points.  Signature and semantics recalled from upstream (its source is not in the reference snapshot)."""
from rodygs_b200.knn import dist_cuda2

distCUDA2 = dist_cuda2

__all__ = ["distCUDA2"]
