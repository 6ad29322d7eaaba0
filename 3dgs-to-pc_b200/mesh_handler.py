"""Point-cloud post-processing (reference: mesh_handler.py).

clean_point_cloud runs on the GPU (g2pc/outliers.py, csrc/s9_knn.cu) with the semantics of the reference's Open3D call.
Meshing (Open3D Poisson reconstruction, Laplacian smoothing) is not part of this build: generate_mesh fails with a
clear message."""
import torch

from g2pc import outliers


def clean_point_cloud(points, colours, normals, std_ratio=10, device="cuda:0"):
    """Drop statistical outliers: Open3D's remove_statistical_outlier(nb_neighbors=20, std_ratio) as the reference calls
    it (mesh_handler.py:89-94).  Returns (points, colours int32, normals) of the kept rows in their original order.
    Colours come out as int32(clamp(c, 0, 255)), like the reference's round trip through Open3D.  Unlike the reference,
    points and normals keep their input dtype (the reference returns float64 with the same values), and normals None
    stays None (the reference yields an empty (0, 3) tensor).  Points must be float32 (the pipeline's output dtype)."""
    points = points.to(device)
    colours = None if colours is None else torch.clamp(colours.to(device), min=0, max=255).to(torch.int32)
    normals = None if normals is None else normals.to(device)
    index, _ = outliers.select_inliers(points, nb_neighbors=20, std_ratio=std_ratio)
    pts, cols, nrm = outliers.gather_rows(index, [points, colours, normals])
    return pts, cols, nrm


def _need_open3d():
    try:
        import open3d  # noqa: F401
    except ImportError as e:
        raise ImportError("Open3D is required for meshing and is not part of g2pc") from e
    raise NotImplementedError("Open3D meshing is outside the scope of the g2pc hot path")


def generate_mesh(points, colours, normals, output_path, depth=10, laplacian_iters=10):
    _need_open3d()
