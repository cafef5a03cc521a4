"""A minimal stand-in for pytorch3d: only ``pytorch3d.ops.knn_points`` (from opengaussian_b200.knn).  Put ``compat/knn``
on PYTHONPATH only where pytorch3d itself is not installed (see INTEGRATION.md)."""
