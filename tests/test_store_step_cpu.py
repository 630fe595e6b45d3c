"""CPU-side checks of the store tuning steps: the declared prototypes and the argument / geometry checks that run before any
CUDA call."""
import ctypes

STORE_STEP_ARGS = ['raw_store', 'raw_bytes_per_code', 'F', 'gt_store', 'G', 'H', 'W', 'pos', 'N', 'white_level', 'status',
                   'h', 'w', 'loss_out', 'dparams', 'dm_kind', 'dm_clip_hi', 'ops', 'param_off', 'iarg', 'S', 'params',
                   'param_stride', 'P', 'workspace', 'workspace_bytes', 'stream']
NAMES = ('risp_pipeline_mse_step_store', 'risp_pipeline_l1_step_store')


def _lib():
    from reconfigisp_b200 import _build, _lib as L
    lib = ctypes.CDLL(_build.LIB)
    lib.risp_last_error.restype = ctypes.c_char_p
    for name in NAMES:
        fn = getattr(lib, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [t for t, _ in L.PROTOS[name][1]]
    return lib, L


def test_store_steps_are_declared_and_exported():
    from reconfigisp_b200 import _lib as L
    lib, _ = _lib()
    for name in NAMES:
        assert [a for _, a in L.PROTOS[name][1]] == STORE_STEP_ARGS, name
        assert hasattr(lib, name)
    # the step arguments after the store's are those of risp_pipeline_mse_step without raw, gt, y_out and the geometry
    step = [a for _, a in L.PROTOS['risp_pipeline_mse_step'][1]]
    assert STORE_STEP_ARGS[13:] == [a for a in step if a not in ('raw', 'gt', 'y_out', 'N', 'H', 'W')]


def test_store_steps_reject_bad_arguments_and_geometry_without_a_gpu():
    """Null / out-of-range store arguments are RISP_E_INVALID; frames with W % 16 != 0, crops with w % 4 != 0 or odd h and
    unaligned stores are RISP_E_UNSUPPORTED -- all before any CUDA call."""
    lib, L = _lib()
    fake = ctypes.c_void_p(1 << 20)            # 16-byte aligned, never dereferenced: validation fails first
    odd = ctypes.c_void_p((1 << 20) + 4)
    ops_, off, iarg = L.iarr([L.ENUMS['RISP_OP_GAMMA']]), L.iarr([0]), L.iarr([0])

    for name in NAMES:
        def step(raw=fake, bpc=2, F=2, gt=fake, G=2, H=32, W=64, pos=fake, N=2, wl=1023., status=fake, h=16, w=32, loss=fake):
            return getattr(lib, name)(raw, bpc, F, gt, G, H, W, pos, N, wl, status, h, w, loss, fake, 1, 1.0, ops_, off, iarg,
                                      1, fake, 0, 1, fake, 1 << 20, None)

        for kw in (dict(raw=None), dict(gt=None), dict(pos=None), dict(status=None), dict(loss=None), dict(bpc=4), dict(F=0),
                   dict(G=-1), dict(N=0), dict(N=70000), dict(h=2), dict(w=0), dict(h=34), dict(w=80), dict(wl=0.),
                   dict(F=1 << 30, H=4000, W=4000)):
            rc = step(**kw)
            assert rc == L.RISP_E_INVALID, (name, kw, rc)
            assert name.encode() in lib.risp_last_error(), kw
        for kw in (dict(W=56), dict(w=30), dict(h=15), dict(raw=odd), dict(gt=odd), dict(pos=odd)):
            rc = step(**kw)
            assert rc == L.RISP_E_UNSUPPORTED, (name, kw, rc)
            assert name.encode() in lib.risp_last_error(), kw
