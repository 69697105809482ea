from .knn import knn_gather, knn_points  # noqa: F401
from .mesh_face_areas_normals import mesh_face_areas_normals  # noqa: F401
from .points_normals import estimate_pointcloud_local_coord_frames, estimate_pointcloud_normals  # noqa: F401
