from .knn import knn_gather, knn_points  # noqa: F401
from .mesh_face_areas_normals import mesh_face_areas_normals  # noqa: F401
