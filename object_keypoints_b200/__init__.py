"""object_keypoints_b200 -- B200-native (sm_100a) heatmap -> 3D keypoint path of
ethz-asl/object_keypoints, behind the reference's pipeline API.

    from object_keypoints_b200 import ObjectKeypointPipeline, camera_utils
    pipeline = ObjectKeypointPipeline([64, 64], None, {'keypoint_config': [1, 3]})
    pipeline.reset(camera_utils.from_calibration('config/calibration.yaml').scale(...))
    objects = pipeline(heatmap, depth, centers)              # reference semantics, batch 1
    tables = pipeline.decode_batch(heatmaps, depths, centers)  # any batch, stays on the GPU

Importing the package does not need a GPU; constructing a pipeline does (no CPU fallback).
"""
from . import camera_utils, linalg                                   # noqa: F401
from .pipeline import (CameraTable, DecodeTables, StereoTables, SequenceObjectTables, KeypointDecoder, InferenceComponent, KeypointExtractionComponent,   # noqa: F401
                       ObjectExtraction, DetectionToPoint, ObjectKeypointPipeline,
                       LearnedKeypointTrackingPipeline, tables_to_objects, tables_to_keypoints)
from .triangulation import (TriangulationComponent, triangulate, triangulate_multiview, triangulate_stereo,   # noqa: F401
                            undistort_points, project_points, reprojection_filter, correct_matches, associate,
                            AssociationComponent, triangulate_stereo_objects)
from . import evaluation, producer, sharding, targets                # noqa: F401,E402

__version__ = "0.1.0"
