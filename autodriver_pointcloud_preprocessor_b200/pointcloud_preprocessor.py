"""Drop-in counterpart of ``autodriver_pointcloud_preprocessor/pointcloud_preprocessor.py``.

Same class name, constructor, parameter names / defaults / types (``pp.py:129-199``), topics,
method names and ``processing_times`` keys; the per-scan work runs on the GPU through the
C-ABI library.  Two execution paths sit behind ``preprocess()``:

* fused  - one ``apc_pipeline_run`` over the uploaded message bytes (front end -> voxel ->
           statistical -> radius -> RANSAC), no host round trips; carries x, y, z and
           intensity.  Used when the cloud has no other known attribute (ring / time /
           return_type / rgb) or when ``fused_pipeline`` is forced on.
* staged - the reference's own sequence of carrier calls (``pp.py:447-544``) on
           ``geometry.PointCloud``, every attribute gathered / voxel-averaged like Open3D does.

Additive parameters (the reference only has a TODO for radius outlier removal, ``pp.py:37``):
``remove_radius_outliers`` (False), ``.nb_points`` (5), ``.search_radius`` (0.5),
``remove_ground.seed`` (0), ``fused_pipeline`` ('auto').

Duplicate removal follows the back end the reference would pick (``pp.py:452-460``): numpy ->
sorted unique rows, torch -> ``points[inverse]`` exactly as ``utils.py:538-542`` is written
(N rows), anything else -> Open3D semantics; all three run on the device.
Normal estimation (``estimate_normals``, default True like the reference) runs on the device
(``apc_estimate_normals``) and adds ``normal_x/y/z`` to the published cloud (pp.py:560-567).
``save_pointcloud`` writes uncompressed PCD files of the published layout (``pointcloud_loader``).
Deliberate deviations, all visible: visualisation and the other file formats need Open3D and are
skipped with a warning.
"""
from __future__ import annotations

import os
from functools import partial

import numpy as np

np.set_printoptions(suppress=True)

try:
    import scipy
    from scipy.spatial.transform import Rotation as R
    SCIPY_INSTALLED = True
    SCIPY_VERSION = scipy.__version__
except ImportError:  # pragma: no cover
    SCIPY_INSTALLED = False
    SCIPY_VERSION = '0.0.0'

import torch

from . import _capi, engine, geometry
from . import geometry as o3d
from . import geometry as o3c
from ._ros_compat import (HAVE_ROS, Buffer, ConnectivityException, Duration, ExtrapolationException, Header,  # noqa: F401
                          LookupException, Node, Parameter, ParameterDescriptor, ParameterType, PointCloud2,
                          PointField, QoSHistoryPolicy, QoSProfile, QoSReliabilityPolicy, SetParametersResult,
                          Time, TransformListener, point_cloud2, rclpy, tf2_ros)
from .utils import (raw_column, packed_message_bytes, device_native_endian, FIELD_DTYPE_MAP, FIELD_DTYPE_MAP_INV, VENDOR_MAPPINGS, check_field,  # noqa: F401
                    convert_pointcloud_to_numpy, crop_pointcloud, dict_to_open3d_tensor_pointcloud,
                    extract_rgb_from_pointcloud, get_current_time, get_fields_from_dicts, get_pointcloud_metadata,
                    get_time_difference, numpy_struct_to_pointcloud2, pointcloud_to_dict, remove_duplicates,
                    rgb_int_to_float)

PT = ParameterType

#: (name, default, ParameterType) in the reference's declaration order (pp.py:129-199)
PARAMETERS = [
    ('input_topic', "/velodyne_front/velodyne_points", PT.PARAMETER_STRING),
    ('output_topic', "/lidar1/velodyne_points/processed", PT.PARAMETER_STRING),
    ('qos', "SENSOR_DATA", PT.PARAMETER_STRING),
    ('pointcloud_fields', [], None),
    ('queue_size', 1, None),
    ('use_gpu', False, None),
    ('cpu_backend', 'torch', None),
    ('gpu_backend', 'open3d', None),
    ('robot_frame', '', None),
    ('static_camera_to_robot_tf', True, None),
    ('transform_timeout', 0.1, None),
    ('offset_pointcloud_matrix', np.eye(4).flatten().tolist(), None),
    ('offset_pointcloud_frame', '', None),
    ('organize_cloud', False, None),
    ('save_pointcloud', False, None),
    ('pointcloud_save_directory', './pointclouds/', None),
    ('pointcloud_save_prepend_str', '', None),
    ('pointcloud_save_extension', '.pcd', None),
    ('pointcloud_save_ascii', False, None),
    ('pointcloud_save_compressed', False, None),
    ('remove_duplicates', True, None),
    ('remove_nans', True, None),
    ('remove_infs', True, None),
    ('crop_to_roi', True, None),
    ('crop_to_roi.invert', False, None),
    ('roi_min', [-60.0, -60.0, -20.0], None),
    ('roi_max', [60.0, 60.0, 20.0], None),
    ('voxel_size', 0.01, None),
    ('remove_statistical_outliers', False, None),
    ('remove_statistical_outliers.nb_neighbors', 20, None),
    ('remove_statistical_outliers.std_ratio', 2.0, None),
    ('estimate_normals', True, None),
    ('estimate_normals.search_radius', 0.1, None),
    ('estimate_normals.max_neighbors', 30, None),
    ('remove_ground', False, None),
    ('remove_ground.distance_threshold', 0.2, None),
    ('remove_ground.ransac_number', 5, None),
    ('remove_ground.num_iterations', 100, None),
    ('remove_ground.probability', 0.99, None),
    ('ground_plane', [0.0, 1.0, 0.0, 0.0], None),
    ('use_height', True, None),
    ('override_header', False, None),
    ('override_header.stamp_source', 'latest', None),
    ('visualize', False, None),
    ('visualize.window_name', 'Open3D', None),
    ('visualize.window_width', 1920, None),
    ('visualize.window_height', 1080, None),
    ('visualize.zoom', 0.0, None),
    ('visualize.front', [], None),
    ('visualize.lookat', [], None),
    ('visualize.up', [], None),
    ('visualize.save_visualizer_image', False, None),
    ('visualize.visualizer_image_path', './images', None),
]

#: parameters this implementation adds (never renames a reference parameter)
EXTRA_PARAMETERS = [
    ('remove_radius_outliers', False, None),
    ('remove_radius_outliers.nb_points', 5, None),
    ('remove_radius_outliers.search_radius', 0.5, None),
    ('remove_ground.seed', 0, None),
    ('fused_pipeline', 'auto', None),
]

PROCESSING_TIME_KEYS = ['crop', 'ground_segmentation', 'normal_estimation', 'point_clearing', 'pointcloud_msg_parsing',
                        'pointcloud_pub', 'preprocessing_time', 'remove_duplicate_points', 'remove_nan_points',
                        'remove_statistical_outliers', 'ros_to_numpy', 'tensor_transfer', 'tf_lookup',
                        'total_callback_time', 'transform', 'voxel_downsampling']


class PointcloudPreprocessorNode(Node):
    def __init__(self, node_name='pointcloud_preprocessor', enabled=True, parameter_namespace='', **node_kwargs):
        super(PointcloudPreprocessorNode, self).__init__(node_name, **node_kwargs)
        if parameter_namespace:
            parameter_namespace = f'{parameter_namespace.rstrip(".")}.'
        self.parameter_namespace = parameter_namespace

        # Declare parameters (pp.py:129-199)
        for name, default, ptype in PARAMETERS + EXTRA_PARAMETERS:
            if ptype is not None:
                self.declare_parameter(name=f'{self.parameter_namespace}{name}', value=default,
                                       descriptor=ParameterDescriptor(description='', type=ptype))
            else:
                self.declare_parameter(f'{self.parameter_namespace}{name}', default)

        def gp(name):
            return self.get_parameter(f'{self.parameter_namespace}{name}').value

        # Get parameters (pp.py:213-269)
        self.use_sim_time = self.get_parameter('use_sim_time').get_parameter_value().bool_value
        self.input_topic = gp('input_topic')
        self.output_topic = gp('output_topic')
        self.qos = self.get_parameter(f'{self.parameter_namespace}qos').get_parameter_value().string_value
        self.pointcloud_fields = gp('pointcloud_fields')
        self.queue_size = gp('queue_size')
        self.use_gpu = gp('use_gpu')
        self.cpu_backend = gp('cpu_backend')
        self.gpu_backend = gp('gpu_backend')
        self.robot_frame = gp('robot_frame')
        if self.robot_frame:
            assert SCIPY_INSTALLED
            self.rotation_object = None
            self.homogenous_matrix = np.eye(4)
        self.static_camera_to_robot_tf = gp('static_camera_to_robot_tf')
        self.transform_timeout = gp('transform_timeout')
        self.offset_pointcloud_frame = gp('offset_pointcloud_frame')
        self.organize_cloud = gp('organize_cloud')
        self.save_pointcloud = gp('save_pointcloud')
        self.pointcloud_save_directory = gp('pointcloud_save_directory')
        if self.save_pointcloud:
            os.makedirs(self.pointcloud_save_directory, exist_ok=True)
        if not self.pointcloud_save_directory:
            self.pointcloud_save_directory = '.'
        self.pointcloud_save_prepend_str = gp('pointcloud_save_prepend_str')
        self.pointcloud_save_extension = gp('pointcloud_save_extension')
        self.pointcloud_save_ascii = gp('pointcloud_save_ascii')
        self.pointcloud_save_compressed = gp('pointcloud_save_compressed')

        self.remove_duplicates = bool(gp('remove_duplicates'))
        self.remove_nans = bool(gp('remove_nans'))
        self.remove_infs = bool(gp('remove_infs'))
        self.crop_to_roi = gp('crop_to_roi')
        self.crop_to_roi_invert = gp('crop_to_roi.invert')
        self.roi_min = gp('roi_min')
        self.roi_max = gp('roi_max')
        self.voxel_size = gp('voxel_size')
        self.remove_statistical_outliers = gp('remove_statistical_outliers')
        self.remove_statistical_outliers_nb_neighbors = int(gp('remove_statistical_outliers.nb_neighbors'))
        self.remove_statistical_outliers_std_ratio = float(gp('remove_statistical_outliers.std_ratio'))
        self.estimate_normals = gp('estimate_normals')
        self.estimate_normals_search_radius = float(gp('estimate_normals.search_radius'))
        self.estimate_normals_max_neighbors = int(gp('estimate_normals.max_neighbors'))
        self.remove_ground = gp('remove_ground')
        self.remove_ground_distance_threshold = float(gp('remove_ground.distance_threshold'))
        self.remove_ground_ransac_number = int(gp('remove_ground.ransac_number'))
        self.remove_ground_num_iterations = int(gp('remove_ground.num_iterations'))
        self.remove_ground_probability = float(gp('remove_ground.probability'))
        self.ground_plane = gp('ground_plane')
        self.use_height = gp('use_height')
        self.override_header = gp('override_header')
        if self.override_header:
            self.new_header_data = {'frame_id': self.robot_frame, 'stamp_source': gp('override_header.stamp_source')}
        self.visualize = gp('visualize')
        # additive
        self.remove_radius_outliers = gp('remove_radius_outliers')
        self.remove_radius_outliers_nb_points = int(gp('remove_radius_outliers.nb_points'))
        self.remove_radius_outliers_search_radius = float(gp('remove_radius_outliers.search_radius'))
        self.remove_ground_seed = int(gp('remove_ground.seed'))
        self.fused_pipeline = gp('fused_pipeline')

        # Setup the device (pp.py:272-280).  Compute always happens on the GPU; ``use_gpu`` only
        # decides where the carrier keeps its tensors between calls, like the reference's device.
        if not torch.cuda.is_available():
            raise RuntimeError("CUDA device required: this implementation has no CPU path")
        self.torch_device = torch.device('cpu')
        self.o3d_device = o3d.Device('CPU:0')
        if self.use_gpu:
            self.torch_device = torch.device('cuda:0')
            self.o3d_device = o3d.Device('CUDA:0')

        self.offset_pointcloud_matrix = np.array(gp('offset_pointcloud_matrix')).reshape(4, 4)
        if np.allclose(self.offset_pointcloud_matrix, np.eye(4)):
            self.offset_pointcloud_matrix = None
        else:
            self.offset_pointcloud_matrix = o3c.Tensor(self.offset_pointcloud_matrix, dtype=o3c.float32,
                                                       device=self.o3d_device)

        # Initialize variables (pp.py:290-322)
        self.camera_to_robot_tf = None
        self.pointcloud_dictionary = {'header': None, 'positions': None}
        self.frame_count = 0
        self.tf_broadcaster = tf2_ros.TransformBroadcaster(self)
        self.tf_buffer = Buffer()
        self.tf_listener = TransformListener(self.tf_buffer, self)
        self.o3d_pointcloud = o3d.PointCloud(self.o3d_device)
        if self.crop_to_roi:
            min_bound = o3c.Tensor(self.roi_min, dtype=o3c.Dtype.Float32)
            max_bound = o3c.Tensor(self.roi_max, dtype=o3c.Dtype.Float32)
            self.crop_aabb = o3d.AxisAlignedBoundingBox(min_bound, max_bound).to(self.o3d_device)
            self.passthrough_filter = partial(crop_pointcloud, min_bound=self.roi_min, max_bound=self.roi_max,
                                              invert=self.crop_to_roi_invert, aabb=self.crop_aabb)
        self.pointcloud_metadata = None
        self.pointfields, self.point_offset, self.new_dtype = None, None, None
        self.reset_fields = False
        self.processing_times = {}
        self._raw_dev = None            # uploaded message bytes of the current scan
        self._raw_msg = None
        self._warned = set()

        # setup QoS (pp.py:325-335)
        self.qos_profile = QoSProfile(reliability=QoSReliabilityPolicy.RELIABLE, history=QoSHistoryPolicy.KEEP_LAST,
                                      depth=self.queue_size)
        if self.qos.lower() == "sensor_data":
            self.qos_profile = QoSProfile(reliability=QoSReliabilityPolicy.BEST_EFFORT,
                                          history=QoSHistoryPolicy.KEEP_LAST, depth=self.queue_size)

        if self.visualize:
            self._warn_once("visualize=True needs the Open3D GUI; visualisation is skipped")

        self.enabled = enabled
        if self.enabled:
            self.add_on_set_parameters_callback(self.parameter_change_callback)
            self.poincloud_sub = self.create_subscription(PointCloud2, self.input_topic, self.callback,
                                                          qos_profile=self.qos_profile)
            self.pointcloud_pub = self.create_publisher(PointCloud2, self.output_topic, self.queue_size)
            self.get_logger().info(f"{self.get_fully_qualified_name()} node started on device: {self.o3d_device}")

    # ------------------------------------------------------------------------------------------------
    def _warn_once(self, msg):
        if msg not in self._warned:
            self._warned.add(msg)
            self.get_logger().warn(msg)

    def _backend(self):
        """Back-end string the reference would pass on (pp.py:452-460, 496-504)."""
        dev = str(self.o3d_device).lower()
        if 'cpu' in dev:
            return self.cpu_backend
        if 'cuda' in dev or 'gpu' in dev:
            return self.gpu_backend
        return 'open3d'

    def _dedup_mode(self):
        """C-ABI duplicate-removal mode for the back end string of pp.py:452-460."""
        if not self.remove_duplicates:
            return _capi.DEDUP_OFF
        return {'np': _capi.DEDUP_NUMPY, 'numpy': _capi.DEDUP_NUMPY, 'torch': _capi.DEDUP_TORCH_COMPAT,
                'pytorch': _capi.DEDUP_TORCH_COMPAT}.get(self._backend().lower(), _capi.DEDUP_OPEN3D)

    def _use_fused(self):
        if self.fused_pipeline is True or str(self.fused_pipeline).lower() in ('true', '1', 'on'):
            return True
        if self.fused_pipeline is False or str(self.fused_pipeline).lower() in ('false', '0', 'off'):
            return False
        # 'auto': the fused pipeline carries x, y, z, intensity itself, estimates the normals between the
        # outlier and the ground stage, and ring / time / return_type / rgb travel through its index maps.
        # Both paths accept the same parameter ranges (INTEGRATION.md, "Parameter caps").
        return True

    # ------------------------------------------------------------------------------------------------
    def _upload_message(self, ros_cloud):
        """The message's records as one device uint8 buffer.  Tightly packed rows (the usual case) go
        bytes -> a pinned staging buffer kept across frames (one host memcpy) -> one asynchronous copy
        into a device buffer kept across frames; the reference's path through a pageable tensor costs a
        second host copy and a staged transfer (0.50 -> see profiles/node_times.py).  Padded rows
        (row_step > width * point_step) are compacted first, like read_points."""
        n_bytes = ros_cloud.width * ros_cloud.height * ros_cloud.point_step
        tight = int(getattr(ros_cloud, 'row_step', 0) or 0) in (0, ros_cloud.width * ros_cloud.point_step)
        if n_bytes == 0 or not tight or len(ros_cloud.data) < n_bytes:
            return device_native_endian(packed_message_bytes(ros_cloud).cuda(), ros_cloud)
        stage = getattr(self, '_pinned_in', None)
        if stage is None or stage.numel() < n_bytes:
            cap = max(n_bytes + n_bytes // 4, 1 << 20)
            stage = self._pinned_in = torch.empty(cap, dtype=torch.uint8).pin_memory()
            self._dev_in = torch.empty(cap, dtype=torch.uint8, device='cuda')
        stage.numpy()[:n_bytes] = np.frombuffer(ros_cloud.data, dtype=np.uint8, count=n_bytes)
        dev = self._dev_in[:n_bytes]
        dev.copy_(stage[:n_bytes], non_blocking=True)
        return device_native_endian(dev, ros_cloud)       # a no-op unless the message is big-endian

    def extract_pointcloud(self, ros_cloud):
        """pp.py:394-445: message -> device-resident carrier.  Returns None on every path, like
        the reference."""
        try:
            start_time = get_current_time(monotonic=True)
            field_names = self.pointcloud_fields if self.pointcloud_fields else None
            self._raw_msg = ros_cloud
            self._fused_xyzi = None
            n = ros_cloud.width * ros_cloud.height
            # one upload of the message bytes per scan; both paths read this device buffer
            self._raw_dev = self._upload_message(ros_cloud)
            names = tuple(field_names) if field_names else tuple(f.name for f in ros_cloud.fields)
            if not (self.pointcloud_metadata or {}).get('has_intensity', False):
                self.pointcloud_metadata = dict(self.pointcloud_metadata or {}, **get_pointcloud_metadata(names))
            if self._use_fused():
                # fused path: the unpack happens inside the pipeline launch; only metadata is needed here
                self.pointcloud_metadata.update({'header': ros_cloud.header, 'field_names': names,
                                                 'num_fields': len(names)})
                if n == 0:
                    self.get_logger().warn("Received an empty PointCloud. Skipping...")
                    return None
                if not {"x", "y", "z"}.issubset(names):
                    self.get_logger().error("Incoming PointCloud does not have x, y, z fields.")
                    return None
                self.pointcloud_dictionary = {'header': ros_cloud.header, 'positions': None}
                self.processing_times['ros_to_numpy'] = get_time_difference(start_time, get_current_time(monotonic=True))
                self.processing_times['point_clearing'] = 0.0
                self.processing_times['tensor_transfer'] = 0.0
                return None
            self.pointcloud_dictionary, self.pointcloud_metadata = pointcloud_to_dict(
                ros_cloud, field_names, self.remove_nans, self.organize_cloud, self.pointcloud_metadata,
                _data_dev=self._raw_dev)
            cloud_field_names = self.pointcloud_metadata.get('field_names', None)
        except Exception as e:
            self.get_logger().error(f"Failed to convert PointCloud2 message to numpy: {str(e)}")
            return None

        if len(self.pointcloud_dictionary['positions']) == 0:
            self.get_logger().warn("Received an empty PointCloud. Skipping...")
            return None

        if not {"x", "y", "z"}.issubset(cloud_field_names):
            self.get_logger().error("Incoming PointCloud does not have x, y, z fields.")
            return None
        self.processing_times['ros_to_numpy'] = get_time_difference(start_time, get_current_time(monotonic=True))

        start_time = get_current_time(monotonic=True)
        self.o3d_pointcloud.clear()
        self.processing_times['point_clearing'] = get_time_difference(start_time, get_current_time(monotonic=True))

        start_time = get_current_time(monotonic=True)
        if self.pointcloud_metadata.get('has_rgb'):
            rgb = self.pointcloud_dictionary['rgb']
            if check_field('rgb', self.pointcloud_dictionary, self.pointcloud_metadata):
                self.pointcloud_dictionary['rgb'] = o3c.Tensor(rgb.t.to(torch.float32) / 255.0)     # pp.py:429-431
        for key in ('intensity', 'ring', 'time', 'return_type'):
            self.pointcloud_dictionary = get_fields_from_dicts(key, self.pointcloud_dictionary,
                                                               self.pointcloud_metadata)
        self.o3d_pointcloud = dict_to_open3d_tensor_pointcloud(self.pointcloud_dictionary, device=self.o3d_device)
        self.processing_times['tensor_transfer'] = get_time_difference(start_time, get_current_time(monotonic=True))
        return None

    def _transforms(self):
        """The up-to-three transforms of pp.py:480-491, in order, as float32 4x4 arrays."""
        out = []
        off = self.offset_pointcloud_matrix
        if off is not None and self.offset_pointcloud_frame.lower() in ['', 'lidar']:
            out.append(off.t.cpu().numpy())
        if self.camera_to_robot_tf is not None:
            out.append(self.camera_to_robot_tf.t.cpu().numpy())
            if off is not None and self.offset_pointcloud_frame.lower() in 'robot':
                out.append(off.t.cpu().numpy())
        return out

    def preprocess(self):
        """pp.py:447-544."""
        # transform lookup first (needed by both paths; pp.py:475-478)
        start_time = get_current_time(monotonic=True)
        self.get_camera_to_robot_tf(self.pointcloud_metadata["header"].frame_id,
                                    Time.from_msg(getattr(self.pointcloud_metadata["header"], 'stamp', None)))
        self.processing_times['tf_lookup'] = get_time_difference(start_time, get_current_time(monotonic=True))
        if self._use_fused() and self._raw_msg is not None:
            return self._preprocess_fused()
        return self._preprocess_staged()

    def _preprocess_fused(self):
        fused_start_time = get_current_time(monotonic=True)
        msg = self._raw_msg
        n = msg.width * msg.height
        ctx = geometry.get_context(n)
        raw = self._raw_dev
        field_names = self.pointcloud_fields if self.pointcloud_fields else None
        desc = engine.make_cloud_desc(msg.fields, msg.point_step, n, raw, field_names=field_names)
        crop = None
        if self.crop_to_roi:
            mode = {'np': _capi.CROP_NUMPY, 'numpy': _capi.CROP_NUMPY, 'torch': _capi.CROP_TORCH,
                    'pytorch': _capi.CROP_TORCH}.get(self._backend().lower(), _capi.CROP_OPEN3D)
            crop = dict(min=self.roi_min, max=self.roi_max, invert=self.crop_to_roi_invert, mode=mode)
        fcfg = engine.make_filter_cfg(skip_nans=bool(self.remove_nans and not msg.is_dense),
                                      dedup_mode=self._dedup_mode(),
                                      remove_nan=self.remove_nans, remove_inf=self.remove_infs,
                                      transforms=self._transforms(), crop=crop)
        pcfg = engine.make_pipeline_cfg(
            fcfg, voxel_size=self.voxel_size if self.voxel_size > 0.0 else 0.0,
            statistical=dict(nb_neighbors=self.remove_statistical_outliers_nb_neighbors,
                             std_ratio=self.remove_statistical_outliers_std_ratio)
            if self.remove_statistical_outliers else None,
            radius=dict(nb_points=self.remove_radius_outliers_nb_points,
                        radius=self.remove_radius_outliers_search_radius) if self.remove_radius_outliers else None,
            ground=dict(distance_threshold=self.remove_ground_distance_threshold,
                        ransac_n=self.remove_ground_ransac_number, num_iterations=self.remove_ground_num_iterations,
                        probability=self.remove_ground_probability, seed=self.remove_ground_seed)
            if self.remove_ground else None,
            # estimate_normals is ON by default (pp.py:176) and sits between the outlier and the ground stage
            # (pp.py:521-543): one launch chain, the normals travel through the ground selection
            normals=dict(radius=self.estimate_normals_search_radius, max_nn=self.estimate_normals_max_neighbors)
            if self.estimate_normals else None)
        meta = self.pointcloud_metadata
        extra = [k for k in ('ring', 'time', 'return_type', 'rgb') if meta.get(f'has_{k}')]
        maps = None
        if extra or self.estimate_normals:
            out, counts, plane, maps = ctx.pipeline_run_maps([desc], pcfg)
        else:
            out, counts, plane = ctx.pipeline_run([desc], pcfg)
        c = counts.cpu().numpy()                    # the one synchronisation of the pipeline
        if c[_capi.CNT_STATUS] != 0:                # data-dependent device error (key range / capacity): raise it
            ctx.check()
        n_out = int(c[_capi.CNT_OUTPUT])
        pos, inten = ctx.split_xyzi(out, n_out, want_intensity=bool(self.pointcloud_metadata.get('has_intensity')))
        cloud = o3d.PointCloud(self.o3d_device)
        cloud.point['positions'] = pos if self.use_gpu else pos.cpu()
        if inten is not None:
            cloud.point['intensity'] = (inten if self.use_gpu else inten.cpu()).reshape(-1, 1)
        if extra:
            # attributes the kernels do not touch: cut from the message bytes, gathered with the front
            # end's surviving indices, averaged per voxel "in float32 then cast back" like Open3D does
            # for every attribute (pp.py:511), gathered with the rows that survived the later stages
            m_filt, n_vox = int(c[_capi.CNT_FILTERED]), int(c[_capi.CNT_VOXELS])
            rows = raw[:n * msg.point_step].view(n, msg.point_step)
            by_name = {f.name: f for f in msg.fields}
            ref_dtype = {'ring': torch.uint16, 'time': torch.float64, 'return_type': torch.uint8,
                         'rgb': torch.float32}                                                    # utils.py:110-131, pp.py:429-431

            def carry(col):
                """one attribute column (input order) -> the same column of the output cloud"""
                a = ctx.gather(col.contiguous(), maps['src_idx'], m_filt)
                if self.voxel_size > 0.0:
                    mean = ctx.voxel_mean_attr(a.to(torch.float32).contiguous(), maps['p2v'],
                                               counts[_capi.CNT_VOXELS:_capi.CNT_VOXELS + 1], m_filt,
                                               engine.attr_frac_bits(a))[:n_vox]
                    a = mean.to(col.dtype)
                return ctx.gather(a.contiguous(), maps['out_row'], n_out)

            for key in extra:
                if key == 'rgb':
                    # three uint8 channels (separate r/g/b fields, or one packed float32: utils.py:110-119,
                    # 324-345), scaled to float32 [0, 1] like pp.py:429-431, each carried like any attribute
                    if {"r", "g", "b"}.issubset(by_name):
                        chans = [raw_column(rows, by_name[ch]).to(torch.uint8) for ch in ("r", "g", "b")]
                    else:
                        packed = raw_column(rows, by_name["rgb"]).view(torch.int32)
                        chans = [((packed >> sh) & 0xFF).to(torch.uint8) for sh in (16, 8, 0)]
                    a = torch.stack([carry(ch.to(torch.float32) / 255.0) for ch in chans], 1)
                    cloud.point['rgb'] = a if self.use_gpu else a.cpu()
                    continue
                a = carry(raw_column(rows, by_name[meta[f'{key}_field_name']]).to(ref_dtype[key]))
                cloud.point[key] = (a if self.use_gpu else a.cpu()).reshape(-1, 1)
        if self.estimate_normals and maps is not None:
            nrm = maps['normals'][:n_out]
            cloud.point['normals'] = nrm if self.use_gpu else nrm.cpu()
            self.pointcloud_metadata['has_normals'] = True
        self.o3d_pointcloud = cloud
        self._fused_xyzi = (out[:n_out], cloud)       # prepare_pointcloud repacks straight from this
        self.last_counts = c
        self.last_plane = plane.cpu().numpy()
        # the stages ran as ONE launch chain: the reference's per-stage keys (pp.py:463-543) exist for every
        # enabled stage, the time of the whole chain is booked under 'fused_pipeline'
        fused_time = get_time_difference(fused_start_time, get_current_time(monotonic=True))
        for key, on in (('remove_duplicate_points', self.remove_duplicates), ('remove_nan_points', self.remove_nans or self.remove_infs),
                        ('transform', bool(self._transforms())), ('crop', self.crop_to_roi),
                        ('voxel_downsampling', self.voxel_size > 0.0),
                        ('remove_statistical_outliers', self.remove_statistical_outliers),
                        ('normal_estimation', self.estimate_normals), ('ground_segmentation', self.remove_ground)):
            if on:
                self.processing_times[key] = 0.0
        self.processing_times['fused_pipeline'] = fused_time
        return self.o3d_pointcloud

    def _normals_and_ground(self):
        """pp.py:521-543 on the carrier: estimate_normals, then segment_plane + select_by_index."""
        if self.estimate_normals:
            start_time = get_current_time(monotonic=True)
            self.o3d_pointcloud.estimate_normals(radius=self.estimate_normals_search_radius,
                                                 max_nn=self.estimate_normals_max_neighbors)
            self.pointcloud_metadata['has_normals'] = True
            self.processing_times['normal_estimation'] = get_time_difference(start_time, get_current_time(monotonic=True))
        if self.remove_ground:
            start_time = get_current_time(monotonic=True)
            plane_model, inliers = self.o3d_pointcloud.segment_plane(
                distance_threshold=self.remove_ground_distance_threshold,
                ransac_n=self.remove_ground_ransac_number,
                num_iterations=self.remove_ground_num_iterations,
                probability=self.remove_ground_probability, seed=self.remove_ground_seed)
            self.o3d_pointcloud = self.o3d_pointcloud.select_by_index(inliers, invert=True)
            self.last_plane = plane_model.cpu().numpy()
            self.processing_times['ground_segmentation'] = get_time_difference(start_time, get_current_time(monotonic=True))

    def _preprocess_staged(self):
        # Remove duplicate points (pp.py:450-463), with the back end the reference would use.
        if self.remove_duplicates:
            start_time = get_current_time(monotonic=True)
            backend = self._backend()
            self.o3d_pointcloud, dupl_msg = remove_duplicates(self.o3d_pointcloud, backend)
            self.processing_times['remove_duplicate_points'] = get_time_difference(start_time, get_current_time(monotonic=True))

        if self.remove_nans or self.remove_infs:
            start_time = get_current_time(monotonic=True)
            self.o3d_pointcloud, non_finite_masks = self.o3d_pointcloud.remove_non_finite_points(
                remove_nan=self.remove_nans, remove_infinite=self.remove_infs)
            self.processing_times['remove_nan_points'] = get_time_difference(start_time, get_current_time(monotonic=True))

        if self.offset_pointcloud_matrix is not None and self.offset_pointcloud_frame.lower() in ['', 'lidar']:
            self.o3d_pointcloud.transform(self.offset_pointcloud_matrix)
        if self.camera_to_robot_tf is not None:
            start_time = get_current_time(monotonic=True)
            self.o3d_pointcloud.transform(self.camera_to_robot_tf)
            if self.offset_pointcloud_matrix is not None and self.offset_pointcloud_frame.lower() in 'robot':
                self.o3d_pointcloud.transform(self.offset_pointcloud_matrix)
            self.processing_times['transform'] = get_time_difference(start_time, get_current_time(monotonic=True))

        if self.crop_to_roi:
            start_time = get_current_time(monotonic=True)
            self.o3d_pointcloud, crop_msg = self.passthrough_filter(self.o3d_pointcloud, backend=self._backend())
            self.processing_times['crop'] = get_time_difference(start_time, get_current_time(monotonic=True))

        if self.voxel_size > 0.0:
            start_time = get_current_time(monotonic=True)
            self.o3d_pointcloud = self.o3d_pointcloud.voxel_down_sample(self.voxel_size)
            self.processing_times['voxel_downsampling'] = get_time_difference(start_time, get_current_time(monotonic=True))

        if self.remove_statistical_outliers:
            start_time = get_current_time(monotonic=True)
            self.o3d_pointcloud, _ = self.o3d_pointcloud.remove_statistical_outliers(
                nb_neighbors=self.remove_statistical_outliers_nb_neighbors,
                std_ratio=self.remove_statistical_outliers_std_ratio)
            self.processing_times['remove_statistical_outliers'] = get_time_difference(start_time, get_current_time(monotonic=True))

        if self.remove_radius_outliers:
            self.o3d_pointcloud, _ = self.o3d_pointcloud.remove_radius_outliers(
                nb_points=self.remove_radius_outliers_nb_points,
                search_radius=self.remove_radius_outliers_search_radius)

        self._normals_and_ground()
        return self.o3d_pointcloud

    # ------------------------------------------------------------------------------------------------
    def set_fields(self, ros_cloud):
        """pp.py:546-574."""
        orig_field_names = [f.name for f in ros_cloud.fields]
        orig_field_types = [f.datatype for f in ros_cloud.fields]
        self.new_dtype = [(name, FIELD_DTYPE_MAP[datatype]) for name, datatype in zip(orig_field_names, orig_field_types)]
        if self.estimate_normals:                                                   # pp.py:560-567
            orig_field_names.extend(['normal_x', 'normal_y', 'normal_z'])
            orig_field_types.extend([PointField.FLOAT32, PointField.FLOAT32, PointField.FLOAT32])
            self.new_dtype.extend([(n, FIELD_DTYPE_MAP[PointField.FLOAT32]) for n in ('normal_x', 'normal_y', 'normal_z')])
        self.pointfields, self.point_offset = numpy_struct_to_pointcloud2(
            field_names=orig_field_names, field_datatypes=orig_field_types,
            is_dense=self.remove_nans and self.remove_infs)

    def prepare_pointcloud(self, ros_cloud, o3d_pointcloud=None, pointcloud_metadata=None):
        """pp.py:576-625: carrier -> packed structured array with the input's field names/types.
        The records are assembled on the GPU (``apc_repack``) and copied to the host once."""
        if o3d_pointcloud is None:
            o3d_pointcloud = self.o3d_pointcloud
        if not pointcloud_metadata:
            pointcloud_metadata = self.pointcloud_metadata
        if self.pointfields is None or self.reset_fields:
            self.set_fields(ros_cloud)
            self.reset_fields = False
        num_points = len(o3d_pointcloud.point['positions'])
        dtype = np.dtype(self.new_dtype)
        if num_points == 0:
            return np.zeros(0, dtype=dtype)
        ctx = geometry.get_context(num_points)
        gpu = geometry.PointCloud._gpu
        fused = getattr(self, '_fused_xyzi', None)
        if fused is not None and fused[1] is o3d_pointcloud:
            xyzi = fused[0]                               # still on the device from the fused pipeline
        else:
            inten = gpu(o3d_pointcloud.point['intensity']).reshape(-1).to(torch.float32) if 'intensity' in o3d_pointcloud.point else None
            xyzi = ctx.pack_xyzi(gpu(o3d_pointcloud.point['positions']).to(torch.float32), inten)
        source = {'x': (1, None), 'y': (2, None), 'z': (3, None)}
        for key in ('intensity', 'ring', 'time', 'return_type'):
            fname = pointcloud_metadata.get(f'{key}_field_name')
            if fname and check_field(key, self.pointcloud_dictionary, self.pointcloud_metadata) and key in o3d_pointcloud.point:
                source[fname] = (4, None) if key == 'intensity' else (5, gpu(o3d_pointcloud.point[key]).reshape(-1))
        if 'rgb' in o3d_pointcloud.point and 'rgb' in dtype.names:
            # colours float [0,1] -> packed float32 rgb (utils.py:347-356), device side
            c = (gpu(o3d_pointcloud.point['rgb']) * 255).clip(0, 255).to(torch.uint8).to(torch.int32)
            packed = ((c[:, 0] << 16) | (c[:, 1] << 8) | c[:, 2]).view(torch.float32)
            source['rgb'] = (5, packed.contiguous())
        if (self.estimate_normals or pointcloud_metadata.get('has_normals', False)) and 'normal_x' in dtype.names:
            nrm = gpu(o3d_pointcloud.point['normals']).to(torch.float32)           # pp.py:620-624
            for k, name in enumerate(('normal_x', 'normal_y', 'normal_z')):
                source[name] = (5, nrm[:, k].contiguous())
        out_fields = []
        for f in self.pointfields:
            src, attr = source.get(f.name, (0, None))
            out_fields.append((f.offset, f.datatype, src, attr))
        raw = ctx.repack(xyzi, out_fields, self.point_offset)
        # ONE device -> host copy, into a pinned staging buffer that is kept across frames (two of them,
        # alternating: the array handed out for frame k stays valid while frame k + 1 is prepared);
        # create_cloud copies the records into the message (pp.py:769), so no further host copy is made
        nbytes = num_points * self.point_offset
        slot = self.frame_count & 1
        stage = getattr(self, '_pinned_out', None)
        if stage is None:
            stage = self._pinned_out = [None, None]
        if stage[slot] is None or stage[slot].numel() < nbytes:
            stage[slot] = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8).pin_memory()
        stage[slot][:nbytes].copy_(raw[:nbytes], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return np.frombuffer(stage[slot].numpy(), dtype=dtype, count=num_points)

    def create_header(self, ros_cloud, frame_id=None):
        """pp.py:628-641."""
        new_header = ros_cloud.header
        if frame_id is None:
            pointcloud_frame_id = ros_cloud.header.frame_id
            if (self.camera_to_robot_tf is not None) and self.robot_frame and (self.robot_frame != pointcloud_frame_id):
                new_header.frame_id = self.robot_frame
        if self.override_header:
            if self.new_header_data['stamp_source'].lower() == 'latest':
                new_header.stamp = self.get_clock().now().to_msg()
        return new_header

    def callback(self, ros_cloud):
        """pp.py:643-702."""
        if self.pointcloud_pub.get_subscription_count() == 0:
            return
        try:
            callback_start_time = get_current_time(monotonic=False)
            self.extract_pointcloud(ros_cloud)

            preprocessing_start_time = get_current_time(monotonic=False)
            self.preprocess()
            self.processing_times['preprocessing_time'] = get_time_difference(preprocessing_start_time, get_current_time(monotonic=False))

            start_time = get_current_time(monotonic=True)
            processed_struct = self.prepare_pointcloud(ros_cloud)
            new_header = self.create_header(ros_cloud)
            pc_msg = self.tensor_to_ros_cloud(processed_struct, self.pointfields, header=new_header)
            pc_msg.is_dense = ros_cloud.is_dense and self.remove_nans and self.remove_infs
            self.processing_times['pointcloud_msg_parsing'] = get_time_difference(start_time, get_current_time(monotonic=True))

            start_time = get_current_time(monotonic=True)
            self._last_output_msg = pc_msg
            self.pointcloud_pub.publish(pc_msg)
            self.processing_times['pointcloud_pub'] = get_time_difference(start_time, get_current_time(monotonic=True))

            pcd_number = str(self.frame_count).zfill(8)
            self.pointcloud_saver(pcd_number)
            self.pointcloud_visualizer(pcd_number)
            self.frame_count += 1
            self.processing_times['total_callback_time'] = get_time_difference(callback_start_time, get_current_time(monotonic=False))
        except Exception as e:
            self.get_logger().error(f"Error processing point cloud: {str(e)}")

    def get_camera_to_robot_tf(self, source_frame_id, timestamp=None):
        """pp.py:704-732."""
        if self.camera_to_robot_tf is not None and self.static_camera_to_robot_tf:
            return
        if timestamp is None:
            timestamp = Time()
        if self.robot_frame:
            try:
                transform = self.tf_buffer.lookup_transform(self.robot_frame, source_frame_id, timestamp,
                                                            Duration(seconds=self.transform_timeout))
            except tf2_ros.LookupException as e:
                self.get_logger().error(f"TF Lookup Error: {str(e)}")
                return
            except tf2_ros.ConnectivityException as e:
                self.get_logger().error(f"TF Connectivity Error: {str(e)}")
                return
            except tf2_ros.ExtrapolationException as e:
                self.get_logger().error(f"TF Extrapolation Error: {str(e)}")
                return
            self.camera_to_robot_tf = self.transform_to_matrix(transform)
            return

    def transform_to_matrix(self, transform):
        """pp.py:734-760: TransformStamped -> float32 4x4 carrier tensor."""
        translation = transform.transform.translation
        rotation = transform.transform.rotation
        tx, ty, tz = translation.x, translation.y, translation.z
        qx, qy, qz, qw = rotation.x, rotation.y, rotation.z, rotation.w
        self.rotation_object = R.from_quat([qx, qy, qz, qw])
        self.homogenous_matrix = np.eye(4)
        self.homogenous_matrix[:3, :3] = self.rotation_object.as_matrix()
        self.homogenous_matrix[:3, 3] = [tx, ty, tz]
        return o3c.Tensor(self.homogenous_matrix, dtype=o3c.float32, device=self.o3d_device)

    def tensor_to_ros_cloud(self, cloud_data, fields, header=None):
        """pp.py:762-769."""
        if header is None:
            header = Header()
            header.stamp = self.get_clock().now().to_msg()
        return point_cloud2.create_cloud(header, fields, cloud_data)

    def convert_to_open3d_tensor(self, input_array):
        """pp.py:771-788."""
        if isinstance(input_array, np.ndarray):
            if 'cpu' in str(self.o3d_device).lower():
                return o3c.Tensor.from_numpy(input_array)
            return o3c.Tensor(input_array, device=self.o3d_device)
        if isinstance(input_array, torch.Tensor):
            return o3c.Tensor.from_dlpack(torch.utils.dlpack.to_dlpack(input_array))
        self.get_logger().warn("The input array is neither a numpy ndarray nor a torch tensor. Passing through.")
        return o3c.Tensor(input_array, device=self.o3d_device)

    def copy_fields(self, field_name, pointcloud=None):
        """pp.py:790-812."""
        field_names = [field_name] if isinstance(field_name, str) else field_name
        if pointcloud is None:
            pointcloud = self.o3d_pointcloud
        processed_fields = {}
        for field_name_ in field_names:
            try:
                processed_fields[field_name_] = pointcloud.point[field_name_].cpu().numpy().reshape(-1)
            except KeyError:
                self.get_logger().warn(f"Field name: {field_name_} not found in pointcloud {pointcloud}.",
                                       throttle_duration_sec=60.0)
                processed_fields[field_name_] = None
        if isinstance(field_name, str):
            processed_fields = processed_fields[field_name]
        return processed_fields

    def publish_normals_marker_array(self, pointcloud):
        pass

    # ------------------------------------------------------------------------------------------------
    def parameter_change_callback(self, params):
        """pp.py:817-1004, including its type guards (``offset_pointcloud_matrix`` is guarded by
        DOUBLE and ``pointcloud_save_ascii`` by STRING in the reference, so neither can be set;
        unknown or mistyped parameters give ``successful = False``)."""
        T = Parameter.Type
        result = SetParametersResult()
        result.successful = True
        ns = self.parameter_namespace
        simple = {   # name -> (type guard, attribute)
            'cpu_backend': (T.STRING, 'cpu_backend'), 'gpu_backend': (T.STRING, 'gpu_backend'),
            'static_camera_to_robot_tf': (T.BOOL, 'static_camera_to_robot_tf'),
            'transform_timeout': (T.DOUBLE, 'transform_timeout'),
            'offset_pointcloud_frame': (T.STRING, 'offset_pointcloud_frame'),
            'organize_cloud': (T.BOOL, 'organize_cloud'), 'save_pointcloud': (T.BOOL, 'save_pointcloud'),
            'pointcloud_save_directory': (T.STRING, 'pointcloud_save_directory'),
            'pointcloud_save_prepend_str': (T.STRING, 'pointcloud_save_prepend_str'),
            'pointcloud_save_extension': (T.STRING, 'pointcloud_save_extension'),
            'pointcloud_save_ascii': (T.STRING, 'pointcloud_save_ascii'),
            'pointcloud_save_compressed': (T.BOOL, 'pointcloud_save_compressed'),
            'remove_duplicates': (T.BOOL, 'remove_duplicates'), 'remove_nans': (T.BOOL, 'remove_nans'),
            'remove_infs': (T.BOOL, 'remove_infs'), 'voxel_size': (T.DOUBLE, 'voxel_size'),
            'remove_statistical_outliers': (T.BOOL, 'remove_statistical_outliers'),
            'remove_statistical_outliers.nb_neighbors': (T.INTEGER, 'remove_statistical_outliers_nb_neighbors'),
            'remove_statistical_outliers.std_ratio': (T.DOUBLE, 'remove_statistical_outliers_std_ratio'),
            'estimate_normals.search_radius': (T.DOUBLE, 'estimate_normals_search_radius'),
            'estimate_normals.max_neighbors': (T.INTEGER, 'estimate_normals_max_neighbors'),
            'remove_ground': (T.BOOL, 'remove_ground'),
            'remove_ground.distance_threshold': (T.DOUBLE, 'remove_ground_distance_threshold'),
            'remove_ground.ransac_number': (T.INTEGER, 'remove_ground_ransac_number'),
            'remove_ground.num_iterations': (T.INTEGER, 'remove_ground_num_iterations'),
            'remove_ground.probability': (T.DOUBLE, 'remove_ground_probability'),
            'ground_plane': (T.DOUBLE_ARRAY, 'ground_plane'), 'use_height': (T.BOOL, 'use_height'),
            'visualize': (T.BOOL, 'visualize'),
            # additive parameters
            'remove_radius_outliers': (T.BOOL, 'remove_radius_outliers'),
            'remove_radius_outliers.nb_points': (T.INTEGER, 'remove_radius_outliers_nb_points'),
            'remove_radius_outliers.search_radius': (T.DOUBLE, 'remove_radius_outliers_search_radius'),
            'remove_ground.seed': (T.INTEGER, 'remove_ground_seed'),
            'fused_pipeline': (T.STRING, 'fused_pipeline'),
        }

        def rebuild_filter():
            self.passthrough_filter = partial(crop_pointcloud, min_bound=self.roi_min, max_bound=self.roi_max,
                                              invert=self.crop_to_roi_invert, aabb=self.crop_aabb)

        for param in params:
            name = param.name[len(ns):] if ns and param.name.startswith(ns) else param.name
            ty = param.type_
            if name == 'input_topic' and ty == T.STRING:
                if param.value == self.input_topic:
                    continue
                self.input_topic = param.value
                (self.pointcloud_metadata or {}).pop('has_intensity', None)
                self.poincloud_sub = self.create_subscription(PointCloud2, self.input_topic, self.callback,
                                                              qos_profile=self.qos_profile)
            elif name == 'output_topic' and ty == T.STRING:
                if param.value == self.output_topic:
                    continue
                self.output_topic = param.value
                (self.pointcloud_metadata or {}).pop('has_intensity', None)
                self.pointcloud_pub = self.create_publisher(PointCloud2, self.output_topic, self.queue_size)
            elif name == 'use_gpu' and ty == T.BOOL:
                self.use_gpu = bool(param.value)
                self.torch_device = torch.device('cuda:0' if self.use_gpu else 'cpu')
                self.o3d_device = o3d.Device('CUDA:0' if self.use_gpu else 'CPU:0')
            elif name == 'robot_frame' and ty == T.STRING:
                robot_frame = param.value
                if robot_frame.lower() != self.robot_frame.lower():
                    assert SCIPY_INSTALLED
                    self.camera_to_robot_tf = None
                    self.rotation_object = None
                    self.homogenous_matrix = np.eye(4)
                self.robot_frame = robot_frame
                if hasattr(self, 'new_header_data'):
                    self.new_header_data['stamp_source'] = robot_frame        # as in the reference (pp.py:899)
            elif name == 'offset_pointcloud_matrix' and ty == T.DOUBLE:      # guard as in the reference (pp.py:906)
                m = np.array(param.value).reshape(4, 4)
                self.offset_pointcloud_matrix = None if np.allclose(m, np.eye(4)) else o3c.Tensor(
                    m, dtype=o3c.float32, device=self.o3d_device)
            elif name == 'crop_to_roi' and ty == T.BOOL:
                self.crop_to_roi = param.value
                self.crop_aabb = o3d.AxisAlignedBoundingBox(o3c.Tensor(self.roi_min, dtype=o3c.Dtype.Float32),
                                                            o3c.Tensor(self.roi_max, dtype=o3c.Dtype.Float32))
                rebuild_filter()
            elif name == 'crop_to_roi.invert' and ty == T.BOOL:
                self.crop_to_roi_invert = param.value
                if not hasattr(self, 'crop_aabb'):
                    self.crop_aabb = None
                rebuild_filter()
            elif name in ('roi_min', 'roi_max') and ty == T.DOUBLE_ARRAY:
                roi_ = list(param.value)
                if len(roi_) == 3:
                    if name == 'roi_min':
                        self.roi_min = roi_
                    else:
                        self.roi_max = roi_
                    if not hasattr(self, 'crop_aabb'):
                        self.crop_aabb = None
                    rebuild_filter()          # the reference keeps the stale AABB here (pp.py:946-954)
                else:
                    result.successful = False
                    result.reason = "ROI min/max must be of length 3"
            elif name == 'estimate_normals' and ty == T.BOOL:
                self.estimate_normals = param.value
                self.reset_fields = True
                if not self.estimate_normals and self.pointcloud_metadata:
                    self.pointcloud_metadata.pop('has_normals', None)
            elif name == 'override_header' and ty == T.BOOL:
                self.override_header = param.value
                if self.override_header:
                    self.new_header_data = {
                        'frame_id': self.robot_frame,
                        'stamp_source': self.get_parameter(f'{ns}override_header.stamp_source').value}
            elif name == 'override_header.stamp_source' and ty == T.STRING:
                self.new_header_data['stamp_source'] = param.value
            elif name in simple and ty == simple[name][0]:
                setattr(self, simple[name][1], param.value)
            else:
                result.successful = False
            self.get_logger().info(f"Success = {result.successful} for param {param.name} to value {param.value}")
        return result

    def _reset_callback(self):
        pass

    def pointcloud_saver(self, pcd_number):
        """pp.py:1010-1022.  The reference hands the cloud to Open3D's writers; here the published
        record layout is written as a PCD v0.7 file (binary, or ascii with ``pointcloud_save_ascii``).
        Other extensions and ``compressed`` need Open3D's writers and are skipped with a warning."""
        if self.save_pointcloud:
            pointcloud_extension = self.pointcloud_save_extension.strip('.')
            msg = getattr(self, '_last_output_msg', None)
            if pointcloud_extension.lower() != 'pcd' or self.pointcloud_save_compressed or msg is None:
                self._warn_once(f"save_pointcloud: only uncompressed .pcd is written without Open3D "
                                f"(extension '{pointcloud_extension}', compressed={self.pointcloud_save_compressed}); skipped")
                return
            from .pointcloud_loader import write_pcd
            os.makedirs(self.pointcloud_save_directory, exist_ok=True)
            pcd_file_name = os.path.join(self.pointcloud_save_directory,
                                         f"{self.pointcloud_save_prepend_str}{pcd_number}.{pointcloud_extension}")
            write_pcd(pcd_file_name, msg, binary=not self.pointcloud_save_ascii)

    def pointcloud_visualizer(self, pcd_number):
        """pp.py:1024-1050 (Open3D GUI; outside the GPU hot path)."""
        if self.visualize:
            self._warn_once("visualize=True needs the Open3D GUI; visualisation is skipped")


def main(args=None):
    """pp.py:1052-1063."""
    if not HAVE_ROS:
        raise RuntimeError("ROS 2 (rclpy) is not installed: run the node inside a ROS 2 environment, or drive "
                           "PointcloudPreprocessorNode.callback() directly")
    rclpy.init(args=args)
    pcd_preprocessor = PointcloudPreprocessorNode()
    try:
        rclpy.spin(pcd_preprocessor)
    except (KeyboardInterrupt, SystemExit):
        pcd_preprocessor.get_logger().info("Shutting down node...")
    finally:
        pcd_preprocessor.destroy_node()
        rclpy.shutdown()


if __name__ == '__main__':
    main()
