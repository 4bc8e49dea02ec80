"""Import shim: `from simple_knn._C import distCUDA2` (src/model/rodygs_static.py:17) resolves to the B200-native exact
grid KNN (rodygs_b200/knn.py), so RoDyGS needs no simple-knn build."""
