"""ctypes binding of ``lib/libfluidaudio_b200.so`` (C ABI declared in ``include/fluidaudio_b200.h``).

The library is the product: it is built in-tree by ``__graft_entry__.build()`` / ``make -C fluidaudio_b200/csrc``.
There is no Python or CPU fallback — if the shared object is missing, or no sm_100a device is visible, every
compute entry point raises.  This module never imports anything from ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libfluidaudio_b200.so")

STATUS_NAMES = {
    0: "OK", 1: "INVALID_ARGUMENT", 2: "INDEX_OVERFLOW", 3: "OUTPUT_TOO_SMALL", 4: "ALLOCATION_FAILURE",
    5: "RUNTIME_ERROR", 6: "NO_DEVICE", 7: "CUDA_ERROR", 8: "UNSUPPORTED", 255: "UNKNOWN_ERROR",
}


class FluidAudioError(RuntimeError):
    def __init__(self, status: int, where: str, detail: str = ""):
        self.status = status
        super().__init__(f"{where}: {STATUS_NAMES.get(status, status)}" + (f" — {detail}" if detail else ""))


NO_VALUE = -2 ** 31   # FA_NO_VALUE: an absent optional count (Swift nil)


class MelConfig(C.Structure):
    _fields_ = [("sample_rate", C.c_int32), ("n_mels", C.c_int32), ("n_fft", C.c_int32), ("hop_length", C.c_int32),
                ("win_length", C.c_int32), ("preemph", C.c_float), ("pad_to", C.c_int32), ("log_floor", C.c_float),
                ("log_floor_mode", C.c_int32), ("window_periodic", C.c_int32)]


class AudioFormat(C.Structure):
    _fields_ = [("in_rate", C.c_double), ("out_rate", C.c_double), ("channels", C.c_int32), ("format", C.c_int32),
                ("interleaved", C.c_int32), ("algorithm", C.c_int32)]


class VbxConfig(C.Structure):
    _fields_ = [("Fa", C.c_double), ("Fb", C.c_double), ("max_iterations", C.c_int32), ("epsilon", C.c_double),
                ("init_smoothing", C.c_double)]


class ClusterConfig(C.Structure):
    _fields_ = [("threshold", C.c_double), ("vbx", VbxConfig), ("num_speakers", C.c_int32),
                ("min_speakers", C.c_int32), ("max_speakers", C.c_int32), ("reserved", C.c_int32)]


class ClusterInfo(C.Structure):
    _fields_ = [("training_count", C.c_int32), ("initial_clusters", C.c_int32), ("vbx_iterations", C.c_int32),
                ("centroid_count", C.c_int32), ("ms_normalize", C.c_float), ("ms_ahc", C.c_float),
                ("ms_cut", C.c_float), ("ms_vbx", C.c_float), ("ms_assign", C.c_float), ("ms_total", C.c_float),
                ("was_adjusted", C.c_int32), ("detected_clusters", C.c_int32)]


class ReconstructConfig(C.Structure):
    _fields_ = [("frame_duration", C.c_double), ("window_duration", C.c_double), ("min_gap_duration", C.c_double),
                ("seg_min_duration_off", C.c_double), ("seg_min_duration_on", C.c_double),
                ("min_segment_duration", C.c_double), ("exclusive_segments", C.c_int32), ("reserved", C.c_int32)]


# every symbol include/fluidaudio_b200.h and include/FastClusterWrapper.h declare (tests check the export table)
EXPORTED_SYMBOLS = [
    "fa_version", "fa_last_error", "fa_device_count", "fa_set_device", "fa_device_synchronize",
    "fa_kernel_launch_count", "fa_host_alloc", "fa_host_free", "fa_device_alloc", "fa_device_free", "fa_memcpy_h2d",
    "fa_memcpy_d2h", "fa_memcpy_probe", "fa_timer_start", "fa_timer_stop_ms", "fa_mel_default_config", "fa_mel_create",
    "fa_mel_destroy", "fa_mel_get_window", "fa_mel_get_filterbank", "fa_mel_frame_count", "fa_mel_compute",
    "fa_mel_compute_device", "fa_mel_compute_batch", "fa_mel_compute_batch_device", "fa_mel_timer_start",
    "fa_mel_timer_stop_ms", "fa_mel_set_precision", "fa_mel_get_precision", "fa_mel_set_pipeline_chunks", "fa_mel_set_zero_copy_output", "fa_mel_normalize_per_feature", "fa_mel_unified_features", "fa_mel_lseend_features",
    "fa_resample_output_count", "fa_audio_resample", "fa_audio_to_mel",
    "fa_linear_resample", "fa_l2_normalize_rows", "fa_ahc_cluster", "fa_dendrogram_cut", "fa_vbx_default_config",
    "fa_vbx_refine", "fa_compute_centroids", "fa_assign_embeddings", "fa_cluster_default_config",
    "fa_diarize_cluster", "fa_diarize_cluster_batch", "fa_diarize_cluster_batch_chunks", "fa_ahc_last_stage_ms", "fa_ahc_last_placement", "fa_diarize_cluster_chunks",
    "fa_hungarian_solve", "fa_max_score_assignment", "fa_constrained_assign", "fa_build_chunk_assignments",
    "fa_export_shape", "fa_export_read", "fa_export_write", "fa_kmeans_cluster", "fa_speaker_constraints_resolve",
    "fa_reconstruct_default_config", "fa_build_segments", "fa_build_speaker_database",
    "fastcluster_compute_centroid_linkage",
]

_lib = None


def load():
    """Load the CUDA library, failing loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FluidAudioError(6, "fluidaudio_b200",
                              f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, f32, f64, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_size_t
    L.fa_version.restype = C.c_char_p
    L.fa_last_error.restype = C.c_char_p
    L.fa_device_count.restype = i32
    L.fa_set_device.argtypes = [i32]
    L.fa_kernel_launch_count.restype = i64
    L.fa_host_alloc.argtypes = [sz, C.POINTER(vp)]
    L.fa_host_free.argtypes = [vp]
    L.fa_device_alloc.argtypes = [sz, C.POINTER(vp)]
    L.fa_device_free.argtypes = [vp]
    L.fa_memcpy_h2d.argtypes = [vp, vp, sz]
    L.fa_memcpy_d2h.argtypes = [vp, vp, sz]
    L.fa_memcpy_probe.argtypes = [vp, sz, vp, sz, i32, C.POINTER(f32)]
    L.fa_timer_stop_ms.argtypes = [C.POINTER(f32)]
    L.fa_mel_default_config.argtypes = [C.POINTER(MelConfig)]
    L.fa_mel_default_config.restype = None
    L.fa_mel_create.argtypes = [C.POINTER(MelConfig), C.POINTER(vp)]
    L.fa_mel_destroy.argtypes = [vp]
    L.fa_mel_destroy.restype = None
    L.fa_mel_get_window.argtypes = [vp, vp, sz]
    L.fa_mel_get_filterbank.argtypes = [vp, vp, sz]
    L.fa_mel_frame_count.argtypes = [vp, i64, i32, i64]
    L.fa_mel_frame_count.restype = i64
    L.fa_mel_compute.argtypes = [vp, vp, sz, f32, i32, i64, i32, vp, sz, C.POINTER(i64), C.POINTER(i64)]
    L.fa_mel_compute_device.argtypes = L.fa_mel_compute.argtypes
    L.fa_mel_compute_batch.argtypes = [vp, vp, vp, i32, vp, i32, i32, vp, vp, vp, vp]
    L.fa_mel_compute_batch_device.argtypes = L.fa_mel_compute_batch.argtypes
    L.fa_mel_set_precision.argtypes = [vp, i32]
    L.fa_mel_set_pipeline_chunks.argtypes = [vp, i32]
    L.fa_mel_set_zero_copy_output.argtypes = [vp, i32]
    L.fa_mel_get_precision.argtypes = [vp]
    L.fa_mel_get_precision.restype = i32
    L.fa_mel_timer_start.argtypes = [vp]
    L.fa_mel_timer_stop_ms.argtypes = [vp, C.POINTER(f32)]
    L.fa_mel_normalize_per_feature.argtypes = [vp, i64, i32, i64]
    L.fa_mel_unified_features.argtypes = [vp, vp, sz, sz, vp, sz, C.POINTER(i64), C.POINTER(i32)]
    L.fa_mel_lseend_features.argtypes = [vp, vp, sz, vp, C.POINTER(i64), vp, sz, C.POINTER(i64)]
    L.fa_resample_output_count.argtypes = [C.POINTER(AudioFormat), i64]
    L.fa_resample_output_count.restype = i64
    L.fa_audio_resample.argtypes = [vp, i64, C.POINTER(AudioFormat), vp, i64, C.POINTER(i64)]
    L.fa_audio_to_mel.argtypes = [vp, vp, i64, C.POINTER(AudioFormat), f32, i32, i32, vp, sz, C.POINTER(i64),
                                  C.POINTER(i64), C.POINTER(i64)]
    L.fa_linear_resample.argtypes = [vp, i64, i32, f64, f64, vp, i64, C.POINTER(i64)]
    L.fa_l2_normalize_rows.argtypes = [vp, sz, sz, vp]
    L.fa_ahc_cluster.argtypes = [vp, sz, sz, f64, vp]
    L.fa_dendrogram_cut.argtypes = [vp, sz, f64, vp]
    L.fa_vbx_default_config.argtypes = [C.POINTER(VbxConfig)]
    L.fa_vbx_default_config.restype = None
    L.fa_vbx_refine.argtypes = [vp, sz, sz, vp, sz, vp, i32, C.POINTER(VbxConfig), vp, vp, vp, vp, C.POINTER(i32)]
    L.fa_compute_centroids.argtypes = [vp, sz, sz, vp, vp, i32, vp, C.POINTER(i32)]
    L.fa_assign_embeddings.argtypes = [vp, sz, sz, vp, i32, vp, vp]
    L.fa_cluster_default_config.argtypes = [C.POINTER(ClusterConfig)]
    L.fa_cluster_default_config.restype = None
    L.fa_diarize_cluster.argtypes = [vp, vp, sz, sz, sz, vp, C.POINTER(ClusterConfig), vp, vp, vp, i32,
                                     C.POINTER(ClusterInfo)]
    L.fa_diarize_cluster_batch.argtypes = [vp, vp, vp, i32, sz, sz, vp, C.POINTER(ClusterConfig), vp, vp]
    L.fa_diarize_cluster_batch_chunks.argtypes = [vp, vp, vp, i32, sz, sz, vp, C.POINTER(ClusterConfig), vp, vp, vp]
    L.fa_diarize_cluster_chunks.argtypes = [vp, vp, sz, sz, sz, vp, C.POINTER(ClusterConfig), vp, vp, vp, vp, i32,
                                            C.POINTER(ClusterInfo)]
    L.fa_hungarian_solve.argtypes = [vp, i32, vp]
    L.fa_max_score_assignment.argtypes = [vp, i32, i32, vp]
    L.fa_constrained_assign.argtypes = [vp, sz, i32, vp, vp]
    L.fa_build_chunk_assignments.argtypes = [vp, vp, vp, sz, i32, i32, i32, vp]
    L.fa_kmeans_cluster.argtypes = [vp, sz, sz, i32, i32, i32, C.c_uint64, vp, vp, i32, C.POINTER(i32), C.POINTER(i32)]
    L.fa_speaker_constraints_resolve.argtypes = [i64, i64, i64, i64, C.POINTER(i64), C.POINTER(i64)]
    L.fa_reconstruct_default_config.argtypes = [C.POINTER(ReconstructConfig)]
    L.fa_reconstruct_default_config.restype = None
    L.fa_build_segments.argtypes = [vp, i32, i32, i32, vp, i32, vp, i32, i32, C.POINTER(ReconstructConfig), vp, vp, vp, vp,
                                    i32, C.POINTER(i32)]
    L.fa_build_speaker_database.argtypes = [vp, i32, vp, i32, i32, vp, vp]
    L.fa_export_shape.argtypes = [C.c_char_p, C.POINTER(sz), C.POINTER(sz), C.POINTER(sz)]
    L.fa_export_read.argtypes = [C.c_char_p, sz, sz, sz, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.fa_export_write.argtypes = [C.c_char_p, sz, sz, sz, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.fa_ahc_last_stage_ms.argtypes = [vp]
    L.fa_ahc_last_stage_ms.restype = None
    L.fa_ahc_last_placement.argtypes = [vp]
    L.fa_ahc_last_placement.restype = None
    L.fastcluster_compute_centroid_linkage.argtypes = [vp, sz, sz, vp, sz]
    L.fastcluster_compute_centroid_linkage.restype = C.c_int
    _lib = L
    return L


def check(status: int, where: str) -> None:
    if status != 0:
        raise FluidAudioError(int(status), where, load().fa_last_error().decode("utf-8", "replace"))


def ptr(a):
    """Raw data pointer of a C-contiguous numpy array (None passes NULL)."""
    return None if a is None else a.ctypes.data


def device_count() -> int:
    return int(load().fa_device_count())


def set_device(ordinal: int) -> None:
    check(load().fa_set_device(ordinal), "fa_set_device")


def synchronize() -> None:
    check(load().fa_device_synchronize(), "fa_device_synchronize")


def kernel_launch_count() -> int:
    return int(load().fa_kernel_launch_count())


class PinnedArray:
    """numpy view over page-locked host memory from fa_host_alloc (so H2D/D2H copies run at link speed)."""

    def __init__(self, shape, dtype):
        self.shape = tuple(int(s) for s in np.atleast_1d(shape))
        self.dtype = np.dtype(dtype)
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        check(load().fa_host_alloc(max(nbytes, 1), C.byref(p)), "fa_host_alloc")
        self._p = p
        buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self._p is not None:
            self.array = None
            load().fa_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class DeviceBuffer:
    """Raw HBM allocation (fa_device_alloc) for the device-resident entry points."""

    def __init__(self, nbytes: int):
        p = C.c_void_p()
        check(load().fa_device_alloc(max(int(nbytes), 1), C.byref(p)), "fa_device_alloc")
        self.ptr = p
        self.nbytes = int(nbytes)

    def upload(self, a: np.ndarray):
        a = np.ascontiguousarray(a)
        check(load().fa_memcpy_h2d(self.ptr, a.ctypes.data, a.nbytes), "fa_memcpy_h2d")

    def download(self, shape, dtype) -> np.ndarray:
        out = np.empty(shape, dtype)
        check(load().fa_memcpy_d2h(out.ctypes.data, self.ptr, out.nbytes), "fa_memcpy_d2h")
        return out

    def free(self):
        if self.ptr is not None:
            load().fa_device_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
