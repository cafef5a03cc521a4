"""``pytorch3d.ops.knn_points`` on the B200 kNN kernel (D = 3, CUDA tensors)."""
from opengaussian_b200.knn import knn_points  # noqa: F401
