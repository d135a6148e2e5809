"""CPU-side checks of the C-ABI library: it builds, loads, and exports every symbol the
header declares (no compute calls -- those need a GPU)."""
import os
import re
import shutil

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def library():
    from pgmorl_b200 import _lib, build
    if shutil.which("nvcc") or os.path.exists(build.NVCC):
        build.build()
    return _lib.lib()


def header_symbols(name="pgmorl_b200.h"):
    src = open(os.path.join(ROOT, "include", name)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pgm_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_all_exported_and_bound(library):
    from pgmorl_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 7
    for s in syms:
        assert hasattr(library, s), f"{s} declared in include/pgmorl_b200.h but not exported"
        assert s in _lib.SIGNATURES, f"{s} has no ctypes signature in pgmorl_b200/_lib.py"
    assert sorted(_lib.SIGNATURES) == syms


def test_diagnostics_live_in_their_own_library(library):
    """The tcgen05 probes are exported by libpgmorl_b200_diag.so only (include/pgmorl_b200_diag.h)."""
    from pgmorl_b200 import _lib
    diag = _lib.diag_lib()
    syms = [s for s in header_symbols("pgmorl_b200_diag.h") if s.startswith(("pgm_tc_", "pgm_ffma2_"))]
    assert sorted(syms) == sorted(_lib.DIAG_SIGNATURES) and len(syms) == 4
    for s in syms:
        assert hasattr(diag, s)
        assert not hasattr(library, s), f"{s} must not be exported by the product library"


def test_n_par_matches_python_layout(library):
    from pgmorl_b200.layout import ENV_SHAPES
    for d in ENV_SHAPES.values():
        assert library.pgm_n_par(d.obs, d.act, d.obj) == d.n_par
    assert library.pgm_n_par(17, 6, 2) == 11150 and library.pgm_n_par(376, 17, 2) == 57828
    # Hopper-v2, Ant, Swimmer (the reference's other launch scripts)
    assert library.pgm_n_par(11, 3, 2) == 10184 and library.pgm_n_par(27, 8, 2) == 12562 and library.pgm_n_par(8, 2, 2) == 9734


def test_offsets_of_the_other_reference_shapes(library):
    """Hopper-v2, Ant and Swimmer: offsets of the 13 tensors, written out (critic head and actor head start right after
    the two 64-wide halves; their sizes follow M and A)."""
    import ctypes
    want = {(11, 3, 2): [0, 704, 768, 4864, 4928, 5632, 5696, 9792, 9856, 9984, 9986, 10178, 10181],
            (27, 8, 2): [0, 1728, 1792, 5888, 5952, 7680, 7744, 11840, 11904, 12032, 12034, 12546, 12554],
            (8, 2, 2): [0, 512, 576, 4672, 4736, 5248, 5312, 9408, 9472, 9600, 9602, 9730, 9732]}
    for (O, A, M), offs in want.items():
        out = (ctypes.c_int * 13)()
        assert library.pgm_param_offsets(O, A, M, out) == 0 and list(out) == offs


def test_tensor_offsets_match_python_layout(library):
    """The offsets state_dict / checkpoint slicing uses (pgmorl_b200/layout.py) are the ones compiled into the kernels."""
    import ctypes
    from pgmorl_b200.layout import ENV_SHAPES, param_layout
    for d in ENV_SHAPES.values():
        out = (ctypes.c_int * 13)()
        assert library.pgm_param_offsets(d.obs, d.act, d.obj, out) == 0
        layout, n = param_layout(d)
        assert [off for off, _ in layout.values()] == list(out) and n == library.pgm_n_par(d.obs, d.act, d.obj)


def test_argument_errors_are_reported_without_a_gpu(library):
    # argument validation happens before any CUDA call
    rc = library.pgm_gae_adv_f32(None, None, None, None, None, None, 0.99, 0.95, None, None, 1, 1, 1, 1, None)
    assert rc == 1 and b"null" in library.pgm_last_error()


def test_minibatch_split_the_reference_would_run_differently_is_rejected(library):
    """S = 100 samples in B = 32 minibatches: the reference's BatchSampler(drop_last=True) yields 33 minibatches of 3 per
    epoch (a2c/storage.py:133-137), not 32 -- refused with a clear message instead of silently taking fewer steps."""
    import ctypes
    from pgmorl_b200._lib import PpoHyper
    buf = (ctypes.c_double * 8)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    hy = PpoHyper()
    rc = library.pgm_ppo_update_f32(p, p, p, p, p, p, 0, p, p, p, 0, p, p, p, 1, 2, 32, ctypes.byref(hy), p, p, 1024, 0,
                                    1, 100, 17, 6, 2, None)
    assert rc == 1 and b"33 minibatches" in library.pgm_last_error()


def _vecnorm_args(buf, **kw):
    """Arguments of pgm_vecnorm_step_f64 for P = 2, N = 4, O = 3, M = 2, every pointer set (host memory: each case below
    is refused before anything is launched, so nothing reads it); kw replaces single arguments by name."""
    a = dict(raw_obs=buf, raw_rew=buf, raw_obj=buf, done=buf, ob_mean=buf, ob_var=buf, ob_count=buf, ret_acc=buf,
             ret_stat=buf, obj_acc=buf, obj_started=buf, obj_mean=buf, obj_var=buf, obj_count=buf, obs_out=buf, obs_ts=12,
             obj_out=buf, obj_ts=8, mask_out=buf, mask_ts=4, gamma=0.99, clipob=10.0, cliprew=10.0, epsilon=1e-8,
             update=1, reset=0, P=2, N=4, O=3, M=2, stream=None)
    a.update(kw)
    return list(a.values())


@pytest.mark.parametrize("kw,msg", [(dict(N=0), b"bad sizes"), (dict(N=129), b"N=129"), (dict(O=0), b"O=0"),
                                    (dict(ob_count=None), b"ob_mean / ob_var / ob_count go together"),
                                    (dict(obj_var=None), b"obj_mean / obj_var / obj_count go together"),
                                    (dict(done=None), b"done flags are required")])
def test_vecnorm_refusals_without_a_gpu(library, kw, msg):
    """K6 refuses sizes outside 1 <= N <= 128, O >= 1, a running-moment triple with a missing member and a step without
    done flags: rc 1 (argument error, not a CUDA error) and a message naming the problem."""
    import ctypes
    buf = ctypes.cast((ctypes.c_double * 64)(), ctypes.c_void_p)
    assert library.pgm_vecnorm_step_f64(*_vecnorm_args(buf, **kw)) == 1
    assert msg in library.pgm_last_error()


def test_vecnorm_rollout_refuses_no_objectives(library):
    """Rollout-slot mode writes reward vectors into the rollout buffer: M = 0 is refused (rc 1) before any launch."""
    import ctypes
    buf = ctypes.cast((ctypes.c_double * 64)(), ctypes.c_void_p)
    rc = library.pgm_vecnorm_rollout_step_f64(buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf, buf,
                                              buf, 12, buf, 8, buf, 4, buf, 4, 0.99, 10.0, 10.0, 1e-8, 1, 2, 4, 3, 0, None)
    assert rc == 1 and b"M=0" in library.pgm_last_error()


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from pgmorl_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.PgmError):
        _lib.lib()
