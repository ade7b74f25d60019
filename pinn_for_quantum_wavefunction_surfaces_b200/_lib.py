"""ctypes binding of libpinn_b200.so (include/pinn_b200.h).  No fallback: a missing library or a
non-B200 device raises."""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libpinn_b200.so"

EXPORTS = [
    "pinn_version", "pinn_theta_size", "pinn_theta_offsets", "pinn_create", "pinn_destroy", "pinn_last_error",
    "pinn_launch_count", "pinn_set_engine", "pinn_get_engine", "pinn_profile_begin", "pinn_profile_collect", "pinn_loss_fwd_bwd", "pinn_fields", "pinn_loss_fwd_bwd_host",
    "pinn_loss_fwd_bwd_tensors", "pinn_mask_from_index_sets", "pinn_measure_fp32_peak", "pinn_step_kernel_clock",
    "pinn_sample", "pinn_adam_step", "pinn_enet_curve", "pinn_grid_reduce", "pinn_spheroidal_reduce", "pinn_trainer_create", "pinn_trainer_destroy",
    "pinn_trainer_load_state", "pinn_trainer_set_batch", "pinn_trainer_run", "pinn_trainer_read", "pinn_trainer_batch",
    "pinn_trainer_stream",
    "pinn_host_timing", "pinn_dp_init", "pinn_dp_connect", "pinn_dp_connect_local", "pinn_dp_enable", "pinn_dp_status", "pinn_dp_set_timeout", "pinn_dp_shutdown",
]


class TrainConfig(ctypes.Structure):
    """pinn_train_config of include/pinn_b200.h"""
    _fields_ = [("variant", ctypes.c_int), ("best_mode", ctypes.c_int), ("history_mean_E", ctypes.c_int),
                ("sc_sampling", ctypes.c_int), ("n", ctypes.c_int64), ("freeze_after", ctypes.c_int64),
                ("best_after", ctypes.c_int64), ("history_capacity", ctypes.c_int64), ("seed", ctypes.c_uint64),
                ("xL", ctypes.c_float), ("xR", ctypes.c_float), ("yL", ctypes.c_float), ("yR", ctypes.c_float),
                ("zL", ctypes.c_float), ("zR", ctypes.c_float), ("RL", ctypes.c_float), ("RR", ctypes.c_float),
                ("cutoff", ctypes.c_float), ("bcutoff", ctypes.c_float), ("grad_mask", ctypes.c_uint32),
                ("lr", ctypes.c_double), ("beta1", ctypes.c_double), ("beta2", ctypes.c_double), ("eps", ctypes.c_double)]


class PinnError(RuntimeError):
    pass


def library_path():
    """The in-tree library; PINN_B200_LIBRARY points development tools (tools/timeline.py) at an instrumented build."""
    return os.environ.get("PINN_B200_LIBRARY") or os.path.join(_HERE, _LIB_NAME)


_lib = None
_lock = threading.Lock()


def lib():
    """Load the shared library (built by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not os.path.exists(path):
            raise PinnError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU fallback)" % path)
        L = ctypes.CDLL(path)
        vp, i32, i64, u32, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint32, ctypes.c_float
        L.pinn_version.restype = i32
        L.pinn_theta_size.restype = i32
        L.pinn_theta_offsets.argtypes = [ctypes.POINTER(i32)]
        L.pinn_theta_offsets.restype = None
        L.pinn_create.argtypes = [i32, ctypes.POINTER(vp)]
        L.pinn_create.restype = i32
        L.pinn_destroy.argtypes = [vp]
        L.pinn_destroy.restype = i32
        L.pinn_last_error.argtypes = [vp]
        L.pinn_last_error.restype = ctypes.c_char_p
        L.pinn_launch_count.argtypes = [vp]
        L.pinn_launch_count.restype = i64
        L.pinn_set_engine.argtypes = [vp, i32]
        L.pinn_set_engine.restype = i32
        L.pinn_get_engine.argtypes = [vp]
        L.pinn_get_engine.restype = i32
        L.pinn_profile_begin.argtypes = [vp]
        L.pinn_profile_begin.restype = i32
        L.pinn_profile_collect.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i32)]
        L.pinn_profile_collect.restype = i32
        L.pinn_loss_fwd_bwd.argtypes = [vp, i32, i64, vp, vp, vp, vp, i32, vp, vp, vp, u32, f32, vp, vp, vp, vp]
        L.pinn_loss_fwd_bwd.restype = i32
        L.pinn_loss_fwd_bwd_tensors.argtypes = [vp, i32, i64, vp, vp, vp, vp, i32, vp, vp, i32, i32, vp, u32, f32, vp, vp, vp, i32, vp]
        L.pinn_loss_fwd_bwd_tensors.restype = i32
        L.pinn_mask_from_index_sets.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp]
        L.pinn_mask_from_index_sets.restype = i32
        L.pinn_measure_fp32_peak.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                             ctypes.POINTER(ctypes.c_double)]
        L.pinn_measure_fp32_peak.restype = i32
        L.pinn_step_kernel_clock.argtypes = [vp, vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
        L.pinn_step_kernel_clock.restype = i32
        L.pinn_fields.argtypes = [vp, i32, i64, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
        L.pinn_fields.restype = i32
        L.pinn_loss_fwd_bwd_host.argtypes = [vp, i32, i64, vp, vp, vp, vp, i32, vp, vp, vp, u32, f32, vp, vp, vp]
        L.pinn_loss_fwd_bwd_host.restype = i32
        u64, f64 = ctypes.c_uint64, ctypes.c_double
        L.pinn_sample.argtypes = [vp, i64, u64, u64, ctypes.POINTER(f32), f32, f32, vp, vp, vp, vp, vp, vp, vp, vp]
        L.pinn_sample.restype = i32
        L.pinn_adam_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, f64, f64, f64, f64, u32,
                                     i32, i64, i32, vp]
        L.pinn_adam_step.restype = i32
        L.pinn_enet_curve.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp, vp]
        L.pinn_enet_curve.restype = i32
        L.pinn_grid_reduce.argtypes = [vp, i32, vp, i32, i32, i32, ctypes.POINTER(f64), f64, vp, vp, vp, vp, vp]
        L.pinn_grid_reduce.restype = i32
        L.pinn_spheroidal_reduce.argtypes = [vp, i32, vp, i32, vp, i32, vp, vp, i32, vp, vp, vp, vp]
        L.pinn_spheroidal_reduce.restype = i32
        L.pinn_trainer_create.argtypes = [vp, ctypes.POINTER(TrainConfig), vp, ctypes.POINTER(vp)]
        L.pinn_trainer_create.restype = i32
        L.pinn_trainer_destroy.argtypes = [vp]
        L.pinn_trainer_destroy.restype = i32
        L.pinn_trainer_load_state.argtypes = [vp, vp, vp, vp, i64]
        L.pinn_trainer_load_state.restype = i32
        L.pinn_trainer_set_batch.argtypes = [vp, vp, vp, vp, vp, vp, vp]
        L.pinn_trainer_set_batch.restype = i32
        L.pinn_trainer_run.argtypes = [vp, i64, i32, i32]
        L.pinn_trainer_run.restype = i32
        L.pinn_trainer_read.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64]
        L.pinn_trainer_read.restype = i32
        L.pinn_trainer_batch.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(vp),
                                         ctypes.POINTER(vp), ctypes.POINTER(vp)]
        L.pinn_trainer_batch.restype = i32
        L.pinn_trainer_stream.argtypes = [vp]
        L.pinn_trainer_stream.restype = vp
        L.pinn_host_timing.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
        L.pinn_host_timing.restype = i32
        L.pinn_dp_init.argtypes = [vp, i32, i32, vp]
        L.pinn_dp_init.restype = i32
        L.pinn_dp_connect.argtypes = [vp, vp]
        L.pinn_dp_connect.restype = i32
        L.pinn_dp_connect_local.argtypes = [vp, ctypes.POINTER(vp)]
        L.pinn_dp_connect_local.restype = i32
        L.pinn_dp_enable.argtypes = [vp, i32]
        L.pinn_dp_enable.restype = i32
        L.pinn_dp_status.argtypes = [vp, ctypes.POINTER(i64)]
        L.pinn_dp_status.restype = i32
        L.pinn_dp_set_timeout.argtypes = [vp, ctypes.c_double]
        L.pinn_dp_set_timeout.restype = i32
        L.pinn_dp_shutdown.argtypes = [vp]
        L.pinn_dp_shutdown.restype = i32
        _lib = L
        return L


def bind_host_to_device_numa(device=0):
    """Pin the calling process to the CPUs that are local to CUDA device `device` (its PCIe root's NUMA node, read from
    /sys/bus/pci/devices/<id>/local_cpulist).  Host buffers allocated and page-locked AFTERWARDS land on that node, so the
    kernels of the *_host entry read them over the device's own PCIe root instead of across the socket interconnect - which
    is what limits 8 ranks streaming their batches at once.  Returns the CPU set, or None when the topology is unknown."""
    import torch
    try:
        pr = torch.cuda.get_device_properties(int(device))
        busid = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % busid) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                lo, hi = part.split("-")
                cpus.update(range(int(lo), int(hi) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if not cpus or cpus == allowed:
            return None
        os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except (OSError, AttributeError, ValueError, RuntimeError, AssertionError):   # no driver / no sysfs entry: leave the affinity alone
        return None


class Handle:
    """One per process/device (SURVEY 8b threading: calls are serialised by stream order)."""
    _cache = {}
    _cache_lock = threading.Lock()

    def __init__(self, device=0):
        self.L = lib()
        self.device = int(device)
        hp = ctypes.c_void_p()
        rc = self.L.pinn_create(self.device, ctypes.byref(hp))
        if rc != 0:
            raise PinnError("pinn_create(device=%d) failed (%d): %s"
                            % (device, rc, self.L.pinn_last_error(None).decode()))
        self.h = hp

    @classmethod
    def get(cls, device=0):
        device = int(device)
        with cls._cache_lock:
            if device not in cls._cache:
                cls._cache[device] = Handle(device)
            return cls._cache[device]

    def check(self, rc, what):
        if rc != 0:
            raise PinnError("%s failed (%d): %s" % (what, rc, self.L.pinn_last_error(self.h).decode()))

    def launch_count(self):
        return int(self.L.pinn_launch_count(self.h))

    ENGINES = {"ffma": 0, "tcgen05": 1}

    def set_engine(self, name):
        """'tcgen05', the one implementation of the fused step kernel the library carries; 'ffma' raises PinnError."""
        self.check(self.L.pinn_set_engine(self.h, self.ENGINES[name]), "pinn_set_engine")

    def get_engine(self):
        return {v: k for k, v in self.ENGINES.items()}[int(self.L.pinn_get_engine(self.h))]

    def measure_fp32_peak(self):
        """-> (FLOP/s of the FP32 FFMA pipe measured now on this device, milliseconds of one timed kernel, SM MHz it ran at)"""
        r, ms, mhz = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
        self.check(self.L.pinn_measure_fp32_peak(self.h, ctypes.byref(r), ctypes.byref(ms), ctypes.byref(mhz)), "pinn_measure_fp32_peak")
        return 2.0 * r.value, ms.value, mhz.value

    def step_kernel_clock(self, stream):
        """-> effective SM clock (MHz) of the last training evaluation enqueued on `stream` (a cudaStream_t as int)"""
        c, ns = ctypes.c_double(), ctypes.c_double()
        self.check(self.L.pinn_step_kernel_clock(self.h, ctypes.c_void_p(stream), ctypes.byref(c), ctypes.byref(ns)), "pinn_step_kernel_clock")
        return c.value / ns.value * 1e3 if ns.value > 0 else 0.0

    def profile_begin(self):
        self.check(self.L.pinn_profile_begin(self.h), "pinn_profile_begin")

    def profile_collect(self):
        """-> (summed step-kernel milliseconds, number of step-kernel launches) since profile_begin."""
        ms, k = ctypes.c_double(), ctypes.c_int()
        self.check(self.L.pinn_profile_collect(self.h, ctypes.byref(ms), ctypes.byref(k)), "pinn_profile_collect")
        return ms.value, k.value

    # ---- data-parallel exchange fused into the reduction kernel (include/pinn_b200.h: pinn_dp_*) ----
    DP_HANDLE_BYTES = 64

    def dp_init(self, rank, world, want_ipc=True):
        """Allocate this rank's exchange buffer; -> its 64-byte IPC handle (bytes) to be all-gathered."""
        buf = ctypes.create_string_buffer(self.DP_HANDLE_BYTES)
        self.check(self.L.pinn_dp_init(self.h, int(rank), int(world), buf if want_ipc else None), "pinn_dp_init")
        return bytes(buf.raw)

    def dp_connect(self, all_handles):
        """all_handles: the ranks' IPC handles in rank order (list of 64-byte strings)."""
        blob = b"".join(all_handles)
        self.check(self.L.pinn_dp_connect(self.h, ctypes.c_char_p(blob)), "pinn_dp_connect")

    def dp_connect_local(self, handles):
        """Same process, one Handle per device: handles in rank order."""
        arr = (ctypes.c_void_p * len(handles))(*[x.h for x in handles])
        self.check(self.L.pinn_dp_connect_local(self.h, arr), "pinn_dp_connect_local")

    def dp_enable(self, on=True):
        self.check(self.L.pinn_dp_enable(self.h, 1 if on else 0), "pinn_dp_enable")

    def dp_status(self):
        """-> number of completed exchanges; raises if a peer timed out."""
        k = ctypes.c_int64()
        self.check(self.L.pinn_dp_status(self.h, ctypes.byref(k)), "pinn_dp_status")
        return int(k.value)

    def dp_set_timeout(self, seconds):
        self.check(self.L.pinn_dp_set_timeout(self.h, float(seconds)), "pinn_dp_set_timeout")

    def dp_shutdown(self):
        self.check(self.L.pinn_dp_shutdown(self.h), "pinn_dp_shutdown")

    def host_timing(self):
        """-> dict(enqueue, wait, copy_out, total) in microseconds for the last pinn_loss_fwd_bwd_host call."""
        a = (ctypes.c_double * 4)()
        self.check(self.L.pinn_host_timing(self.h, a), "pinn_host_timing")
        return {"enqueue": a[0], "wait": a[1], "copy_out": a[2], "total": a[3]}

    def close(self):
        if self.h:
            self.L.pinn_destroy(self.h)
            self.h = None
