"""A PARTIAL pytorch3d: only `pytorch3d.ops.knn_points` / `knn_gather`, for the one call RoDyGS makes
(src/trainer/losses.py:18, :238-239).  With this repository on PYTHONPATH it shadows a real pytorch3d installed
elsewhere; that is deliberate, because pytorch3d has no build for sm_100 under the reference's pinned toolchain and
RoDyGS imports it at module import time.  Everything else pytorch3d offers is absent here."""
