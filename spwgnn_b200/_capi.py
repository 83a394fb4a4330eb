"""ctypes declarations for include/spwgnn.h (the C ABI of libspwgnn.so).

This module only describes the ABI; `spwgnn_b200._lib` binds it to the nvcc-built shared
library and raises if that library is missing -- there is no CPU fallback in the product.
"""
import ctypes as C

N_TENSORS = 22
# (name, shape) in the order of struct SpwParams (include/spwgnn.h)
PARAM_SPECS = (
    [('rm.w%d' % i, s) for i, s in enumerate([(2, 150), (150, 150), (150, 150), (150, 150)])]
    + [('rm.b%d' % i, (150,)) for i in range(4)]
    + [('om.w%d' % i, s) for i, s in enumerate([(2, 100), (100, 100)])]
    + [('om.b%d' % i, (100,)) for i in range(2)]
    + [('rmp.w%d' % i, s) for i, s in enumerate([(350, 150), (150, 150), (150, 100)])]
    + [('rmp.b%d' % i, s) for i, s in enumerate([(150,), (150,), (100,)])]
    + [('omp.w%d' % i, s) for i, s in enumerate([(300, 100), (100, 101)])]
    + [('omp.b%d' % i, s) for i, s in enumerate([(100,), (101,)])]
)
assert len(PARAM_SPECS) == N_TENSORS


class SpwParams(C.Structure):
    _fields_ = [('p', C.c_void_p * N_TENSORS)]


class SpwGraph(C.Structure):
    _fields_ = [
        ('n_towers', C.c_int32), ('n_nodes', C.c_int32), ('n_edges', C.c_int32),
        ('node_off', C.c_void_p), ('in_off', C.c_void_p), ('in_snd', C.c_void_p), ('in_rcv', C.c_void_p),
        ('out_off', C.c_void_p), ('out_pos', C.c_void_p),
    ]


EXPORTS = ['spw_version', 'spw_last_error', 'spw_launch_count', 'spw_profile', 'spw_profile_report', 'spw_ffma_peak', 'spw_tc_selftest', 'spw_tc2_selftest', 'spw_tc_linear', 'spw_csl_linear', 'spw_edges_count', 'spw_edges_fill', 'spw_sample_sizes', 'spw_sample_jenga', 'spw_sample_tower', 'spw_candidates_remove', 'spw_candidates_drop', 'spw_tower_sums', 'spw_workspace_bytes', 'spw_saved_state_layout',
           'spw_workspace_layout_names', 'spw_workspace_layout', 'spw_forward', 'spw_forward_towers_bytes', 'spw_forward_towers', 'spw_bce_grad', 'spw_backward', 'spw_backward_obj', 'spw_backward_rel']


class SpwError(RuntimeError):
    pass


class CApi:
    """Typed view of a loaded libspwgnn shared object."""

    def __init__(self, path):
        self.path = path
        self.dll = C.CDLL(path)
        d = self.dll
        vp, i32, f64 = C.c_void_p, C.c_int32, C.c_double
        d.spw_version.restype = C.c_int
        d.spw_version.argtypes = []
        d.spw_last_error.restype = C.c_char_p
        d.spw_last_error.argtypes = []
        d.spw_launch_count.restype = C.c_longlong
        d.spw_launch_count.argtypes = []
        d.spw_profile.restype = C.c_int
        d.spw_profile.argtypes = [C.c_int]
        d.spw_profile_report.restype = C.c_int
        d.spw_profile_report.argtypes = [C.c_char_p, C.c_size_t]
        d.spw_ffma_peak.restype = C.c_int
        d.spw_ffma_peak.argtypes = [vp, C.c_int, C.c_int, vp]
        d.spw_tc_selftest.restype = C.c_int
        d.spw_tc_selftest.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, vp, vp]
        d.spw_tc2_selftest.restype = C.c_int
        d.spw_tc2_selftest.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, vp, vp]
        d.spw_tc_linear.restype = C.c_int
        d.spw_tc_linear.argtypes = [C.c_int, vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp, vp, vp, C.c_int,
                                    C.c_int, vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_float, C.c_int, vp, vp]
        d.spw_csl_linear.restype = C.c_int
        ll = C.c_longlong
        d.spw_csl_linear.argtypes = [C.c_int, vp, ll, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp, vp, vp, ll, C.c_int, C.c_int, vp, ll,
                                     C.c_int, C.c_int, vp, vp, vp, ll, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, vp, vp]
        d.spw_edges_count.restype = C.c_int
        d.spw_edges_count.argtypes = [vp, vp, i32, i32, i32, f64, C.c_int, vp, vp, vp, vp]
        d.spw_edges_fill.restype = C.c_int
        d.spw_edges_fill.argtypes = [vp, vp, i32, i32, i32, f64, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        d.spw_sample_sizes.restype = C.c_int
        d.spw_sample_sizes.argtypes = [C.c_uint64, i32, i32, i32, vp, vp]
        d.spw_sample_jenga.restype = C.c_int
        d.spw_sample_jenga.argtypes = [C.c_uint64, i32, vp, vp, vp, vp, C.c_int, vp]
        d.spw_sample_tower.restype = C.c_int
        d.spw_sample_tower.argtypes = [C.c_uint64, i32, vp, vp, vp, vp, C.c_int, vp]
        d.spw_candidates_remove.restype = C.c_int
        d.spw_candidates_remove.argtypes = [vp, i32, vp, vp, C.c_int, vp]
        d.spw_candidates_drop.restype = C.c_int
        d.spw_candidates_drop.argtypes = [vp, i32, vp, i32, f64, vp, vp, C.c_int, vp]
        d.spw_tower_sums.restype = C.c_int
        d.spw_tower_sums.argtypes = [vp, vp, i32, vp, vp, vp]
        d.spw_workspace_bytes.restype = C.c_size_t
        d.spw_workspace_bytes.argtypes = [i32, i32, C.c_int]
        d.spw_saved_state_layout.restype = C.c_int
        d.spw_saved_state_layout.argtypes = [i32, i32, C.POINTER(C.c_int64)]
        d.spw_workspace_layout_names.restype = C.c_char_p
        d.spw_workspace_layout_names.argtypes = []
        d.spw_workspace_layout.restype = C.c_int
        d.spw_workspace_layout.argtypes = [i32, i32, C.c_int, C.POINTER(C.c_int64), C.c_int]
        d.spw_forward.restype = C.c_int
        d.spw_forward.argtypes = [C.POINTER(SpwParams), C.POINTER(SpwGraph), vp, vp, vp, vp, C.c_size_t, C.c_int,
                                  C.c_float, C.c_uint64, vp]
        d.spw_forward_towers_bytes.restype = C.c_size_t
        d.spw_forward_towers_bytes.argtypes = [i32, i32]
        d.spw_forward_towers.restype = C.c_int
        d.spw_forward_towers.argtypes = [C.POINTER(SpwParams), C.POINTER(SpwGraph), i32, vp, vp, vp, vp, C.c_size_t, vp]
        d.spw_bce_grad.restype = C.c_int
        d.spw_bce_grad.argtypes = [vp, vp, i32, f64, vp, vp, vp]
        d.spw_backward.restype = C.c_int
        d.spw_backward.argtypes = [C.POINTER(SpwParams), C.POINTER(SpwGraph), vp, vp, vp, C.c_size_t,
                                   C.POINTER(SpwParams), C.c_float, vp]
        d.spw_backward_obj.restype = C.c_int
        d.spw_backward_obj.argtypes = [C.POINTER(SpwParams), C.POINTER(SpwGraph), vp, vp, vp, C.c_size_t, C.c_float, vp, vp]
        d.spw_backward_rel.restype = C.c_int
        d.spw_backward_rel.argtypes = [C.POINTER(SpwParams), C.POINTER(SpwGraph), vp, vp, vp, C.c_size_t, C.c_float, vp, vp, vp]

    def check(self, rc):
        if rc != 0:
            raise SpwError('libspwgnn error %d: %s' % (rc, self.dll.spw_last_error().decode()))

    def workspace_layout(self, n_nodes, n_edges, training):
        """spw_workspace_layout as a dict: array name -> byte offset, plus the sizes listed in include/spwgnn.h."""
        names = self.dll.spw_workspace_layout_names().decode().split(',')
        out = (C.c_int64 * len(names))()
        count = self.dll.spw_workspace_layout(n_nodes, n_edges, int(training), out, len(names))
        if count < 0:
            self.check(count)
        assert count == len(names), (count, len(names))
        return dict(zip(names, [int(v) for v in out]))

    @staticmethod
    def params(ptrs):
        assert len(ptrs) == N_TENSORS
        s = SpwParams()
        for i, p in enumerate(ptrs):
            s.p[i] = p
        return s

    @staticmethod
    def graph(n_towers, n_nodes, n_edges, node_off, in_off, in_snd, in_rcv, out_off, out_pos):
        return SpwGraph(n_towers, n_nodes, n_edges, node_off, in_off, in_snd, in_rcv, out_off, out_pos)
