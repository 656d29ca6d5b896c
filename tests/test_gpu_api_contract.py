"""The argument contract of the eight frame-level entry points -- vet_spatial, vet_transition, vet_analyze, their _host
and their _vectors variants -- through the C ABI: the return code and the exact vet_last_error() text of every refusal,
which calls return VET_OK without touching their outputs, and the order in which the checks run.

Every buffer is a real allocation far larger than the shapes passed, so no case can reach a kernel with bad memory.
The tile limit of the transition kernels and the refusals of the direct regime are tested in test_gpu_thresholds.py
and test_gpu_parity.py."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

F0, U0 = 3, 4      # frames and users of a valid call
NBYTES = 1 << 16   # every output buffer: more than F0 x max(U0, T0) x 8 bytes of both handles below
FILL = 0xA5

# column order of the expectations below
ENTRY_POINTS = ("vet_spatial", "vet_spatial_host", "vet_spatial_vectors", "vet_transition", "vet_transition_host",
                "vet_transition_vectors", "vet_analyze", "vet_analyze_host")

BAD = ("invalid", "bad argument")
MODE = ("invalid", "bad mode")
EMPTY = ("invalid", "Empty vector dictionary")
NULLBUF = ("invalid", "null buffer")
GRID = ("grid", None)   # VET_ERR_UNSUPPORTED "<entry point>: not available for the latitude/longitude grid tiling ..."
NOOP = ("noop", None)   # VET_OK, outputs untouched
RUN = ("run", None)     # VET_OK: a valid call that computes
NA = None               # the entry point has no such argument

# case -> (changes to a valid call, expectation per entry point)
CASES = {
    "null_handle":        (dict(handle=None),                  (BAD,) * 8),
    "negative_F":         (dict(F=-1),                         (BAD,) * 8),
    "negative_U":         (dict(U=-1),                         (BAD,) * 8),
    "bad_dtype":          (dict(dtype=7),                      (BAD, BAD, NA, BAD, BAD, NA, BAD, BAD)),
    "bad_mode":           (dict(mode=5),                       (NA, NA, NA, MODE, MODE, MODE, MODE, MODE)),
    "negative_F_bad_mode": (dict(F=-1, mode=5),                (NA, NA, NA, BAD, BAD, BAD, BAD, BAD)),
    "F0_bad_mode":        (dict(F=0, mode=5),                  (NA, NA, NA, MODE, MODE, MODE, MODE, MODE)),
    "F0":                 (dict(F=0),                          (NOOP,) * 8),
    "F0_null_buffers":    (dict(F=0, null=("in", "sp", "tr")), (NOOP,) * 8),
    "F1":                 (dict(F=1),                          (RUN, RUN, RUN, NOOP, NOOP, NOOP, RUN, RUN)),
    "F1_U0":              (dict(F=1, U=0),                     (EMPTY, EMPTY, EMPTY, NOOP, NOOP, NOOP, EMPTY, EMPTY)),
    "F1_null_transition_entropy": (dict(F=1, null=("tr",)),    (NA, NA, NA, NOOP, NOOP, NOOP, RUN, RUN)),
    "U0":                 (dict(U=0),                          (EMPTY,) * 8),
    "U0_null_input":      (dict(U=0, null=("in",)),            (EMPTY,) * 8),
    "null_input":         (dict(null=("in",)),                 (NULLBUF,) * 8),
    "null_spatial_entropy": (dict(null=("sp",)),               (NULLBUF, NULLBUF, NULLBUF, NA, NA, NA, NULLBUF, NULLBUF)),
    "null_transition_entropy": (dict(null=("tr",)),            (NA, NA, NA, NULLBUF, NULLBUF, NULLBUF, NULLBUF, NULLBUF)),
    "grid_tiling":        (dict(handle="grid"),                (RUN, RUN, GRID, GRID, GRID, GRID, GRID, GRID)),
    "grid_tiling_negative_F": (dict(handle="grid", F=-1),      (BAD, BAD, GRID, GRID, GRID, GRID, GRID, GRID)),
}

PARAMS = [pytest.param(case, ep, i, id=f"{case}-{ep}")
          for case, (_, expect) in CASES.items() for i, ep in enumerate(ENTRY_POINTS) if expect[i] is not NA]


@pytest.fixture(scope="module")
def env():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import viewport_entropy_toolkit_b200 as vet
    from viewport_entropy_toolkit_b200 import _native as N
    handles = {"lattice": vet.Engine(100, 200, [20], vet.EntropyConfig(fov_angle=90.0)),
               "grid": vet.Engine(100, 200, [1], vet.EntropyConfig(), naive_tiles=(30, 30))}
    for eng in handles.values():
        assert max(eng.num_tiles) * F0 * 8 <= NBYTES
    yield N, handles
    for eng in handles.values():
        eng.close()


class Buffers:
    """Input and outputs of one call: device tensors or host arrays, outputs filled with FILL."""

    def __init__(self, host: bool, vectors: bool):
        if vectors:
            v = np.zeros((F0, U0, 3), np.float64)
            v[..., 2] = 1.0
        else:
            v = np.full((F0, U0, 3), 0.5, np.float32)
        self.host = host
        self.inp = v if host else torch.from_numpy(v).cuda()
        self.outs = [np.full(NBYTES, FILL, np.uint8) if host else torch.full((NBYTES,), FILL, dtype=torch.uint8, device="cuda")
                     for _ in range(8)]

    @staticmethod
    def ptr(a):
        return a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr()

    def untouched(self) -> bool:
        torch.cuda.synchronize()
        return all(bool((o == FILL).all()) for o in self.outs)


def _call(N, name, h, b: Buffers, dtype, F, U, mode, null):
    lib = N.load_library()
    inp = None if "in" in null else b.ptr(b.inp)
    o = [b.ptr(x) for x in b.outs]
    sp = [None if "sp" in null else o[0], o[1], o[2], o[3]]  # entropy, per_k, hist0, assign0
    tr = [None if "tr" in null else o[4], o[5], o[6], o[7]]  # entropy, per_k, prev_count0, pairs0
    head = [h, inp] + ([] if name.endswith("_vectors") else [dtype]) + [F, U]
    tail = [] if name.endswith("_host") else [None]  # the legacy default stream
    if name.startswith("vet_spatial"):
        args = head + sp + tail
    elif name.startswith("vet_transition"):
        args = head + tr + [mode] + tail
    else:
        args = head + sp + tr + [mode] + tail
    return getattr(lib, name)(*args)


@pytest.mark.parametrize("case,entry,col", PARAMS)
def test_argument_contract(env, case, entry, col):
    N, handles = env
    changes, expect = CASES[case]
    kind, msg = expect[col]
    handle = changes.get("handle", "lattice")
    h = None if handle is None else handles[handle]._h
    b = Buffers(host=entry.endswith("_host"), vectors=entry.endswith("_vectors"))
    dtype = changes.get("dtype", N.VET_F64 if entry.endswith("_vectors") else N.VET_F32)
    rc = _call(N, entry, h, b, dtype, changes.get("F", F0), changes.get("U", U0),
               changes.get("mode", N.VET_TRANSITION_LITERAL), changes.get("null", ()))
    if kind == "run":
        assert rc == N.VET_OK, N.last_error()
        torch.cuda.synchronize()
        return
    if kind == "noop":
        assert rc == N.VET_OK, N.last_error()
    elif kind == "grid":
        assert rc == N.VET_ERR_UNSUPPORTED
        assert N.last_error() == (f"{entry}: not available for the latitude/longitude grid tiling "
                                  "(the reference has no such path)")
    else:
        assert rc == N.VET_ERR_INVALID_ARG
        assert N.last_error() == msg
    assert b.untouched(), "a call that computes nothing wrote to its outputs"
