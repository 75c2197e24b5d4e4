"""CPU-only: the utility layer of the drop-in boundary (include/libxsmm_utils.h, csrc/host_utils.c) pinned against the
UNMODIFIED reference (oracle/_ref): libxsmm_matdiff statistics and epsilon (the drivers' pass/fail number), matdiff_reduce,
the sequence generator, low-precision array conversions, libxsmm_coprime2 / LIBXSMM_MATINIT (the drivers' input fill).
Where the reference is not built, its stored answers stand in for it (tests/ref_answers.py)."""
import ctypes as C
import os
import subprocess

import numpy as np

import gen
import libxsmm_b200 as X
import ref_answers as R
from oracle_ffi import ref_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L = X.lib
_P, _I, _D = C.c_void_p, C.c_int, C.c_double
if ref_lib is not None:
    ref_lib.ref_matdiff.restype, ref_lib.ref_matdiff.argtypes = _I, [_I, _I, _I, _P, _P, _I, _I, _P]
    ref_lib.ref_matdiff_reduce.restype, ref_lib.ref_matdiff_reduce.argtypes = _I, [_I, _I, _I, _I, _P, _P, _P]
    ref_lib.ref_rng.restype, ref_lib.ref_rng.argtypes = None, [C.c_uint, _P, _I, _P, _I, _P, _I, C.c_uint]
    ref_lib.ref_lp_convert.restype, ref_lib.ref_lp_convert.argtypes = None, [_I, _P, _P, C.c_ulonglong]
    ref_lib.ref_extstate.restype, ref_lib.ref_extstate.argtypes = None, [C.c_uint, _P]
    ref_lib.ref_stochastic_bf8.restype, ref_lib.ref_stochastic_bf8.argtypes = None, [_P, _P, C.c_uint, _P, C.c_uint]
    ref_lib.ref_sexp2_i8i.restype, ref_lib.ref_sexp2_i8i.argtypes = C.c_float, [_I]
    ref_lib.ref_nearbyintf.restype, ref_lib.ref_nearbyintf.argtypes = C.c_float, [C.c_float]
    ref_lib.ref_coprime2.restype, ref_lib.ref_coprime2.argtypes = C.c_ulonglong, [C.c_ulonglong]
    ref_lib.ref_matinit.argtypes = [_I, _D, _P, _I, _I, _I, _D]


class MatdiffInfo(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("norm1_abs norm1_rel normi_abs normi_rel normf_rel linf_abs linf_rel l2_abs l2_rel rsq l1_ref min_ref max_ref "
                                          "avg_ref var_ref l1_tst min_tst max_tst avg_tst var_tst v_ref v_tst").split()] + [(n, C.c_int) for n in "mnir"]


L.libxsmm_matdiff.restype, L.libxsmm_matdiff.argtypes = _I, [C.POINTER(MatdiffInfo), _I, _I, _I, _P, _P, C.POINTER(C.c_int), C.POINTER(C.c_int)]
L.libxsmm_matdiff_epsilon.restype, L.libxsmm_matdiff_epsilon.argtypes = _D, [C.POINTER(MatdiffInfo)]
L.libxsmm_matdiff_reduce.restype, L.libxsmm_matdiff_reduce.argtypes = None, [C.POINTER(MatdiffInfo), C.POINTER(MatdiffInfo)]
L.libxsmm_matdiff_clear.restype, L.libxsmm_matdiff_clear.argtypes = None, [C.POINTER(MatdiffInfo)]


def _image(info):
    return np.array([getattr(info, n) for n, _ in MatdiffInfo._fields_] + [L.libxsmm_matdiff_epsilon(C.byref(info))], dtype=np.float64)


def _same(a, b):
    return np.array_equal(a, b) or np.array_equal(np.nan_to_num(a, nan=-7.0), np.nan_to_num(b, nan=-7.0))


def test_matdiff_matches_reference_bit_for_bit():
    rng = np.random.default_rng(11)
    n_checked = 0
    for dt, npdt in ((gen.F64, np.float64), (gen.F32, np.float32), (gen.I32, np.int32), (gen.I8, np.int8), (14, np.uint8), (gen.I16, np.int16),
                     (gen.BF16, np.uint16), (gen.F16, np.uint16)):
        for (m, n, ldr, ldt) in ((13, 5, 0, 0), (32, 48, 40, 36), (7, 1, 0, 0), (1, 9, 0, 0), (64, 64, 64, 80)):
            lr, lt = (ldr or m), (ldt or m)
            if npdt in (np.float64, np.float32):
                a = rng.standard_normal(lr * n).astype(npdt); b = np.resize(a, lt * n).copy()
                b[:lt * n] = (rng.standard_normal(lt * n) * 1e-3).astype(npdt)
                b.reshape(n, lt)[:, :m] += a.reshape(n, lr)[:, :m]
            elif npdt == np.uint16:
                f = rng.standard_normal(lr * n).astype(np.float32)
                conv = gen.f32_to_bf16_bits if dt == gen.BF16 else (lambda x: np.asarray(x, dtype=np.float32).astype(np.float16).view(np.uint16))
                a = conv(f); b = np.zeros(lt * n, dtype=np.uint16)
                b.reshape(n, lt)[:, :m] = conv((f.reshape(n, lr)[:, :m] * 1.01).astype(np.float32).ravel()).reshape(n, m)
            else:
                a = rng.integers(-100 if npdt != np.uint8 else 0, 100, size=lr * n).astype(npdt); b = np.zeros(lt * n, dtype=npdt)
                b.reshape(n, lt)[:, :m] = a.reshape(n, lr)[:, :m] + (rng.random((n, m)) < 0.1)
            for variant in ("diff", "equal", "nan_tst", "one_sided"):
                aa, bb = a.copy(), b.copy()
                if variant == "equal":
                    bb.reshape(n, lt)[:, :m] = aa.reshape(n, lr)[:, :m]
                if variant == "nan_tst":
                    if npdt not in (np.float64, np.float32):
                        continue
                    bb[(n // 2) * lt + m // 2] = np.nan
                tst_ptr = None if variant == "one_sided" else bb.ctypes.data

                def run_ref():
                    want = np.zeros(28)      # the return code, then the 22 statistics, m n i r and the epsilon
                    want[0] = ref_lib.ref_matdiff(dt, m, n, aa.ctypes.data, tst_ptr, ldr, ldt, want[1:].ctypes.data)
                    return want
                res = R.value(run_ref)
                rc_r, want = int(res[0]), res[1:]
                info = MatdiffInfo()
                plr, plt = C.c_int(ldr), C.c_int(ldt)
                rc_o = L.libxsmm_matdiff(C.byref(info), dt, m, n, aa.ctypes.data, tst_ptr, C.byref(plr) if ldr else None, C.byref(plt) if ldt else None)
                assert rc_o == rc_r
                got = _image(info)
                assert _same(got, want), (dt, m, n, ldr, ldt, variant, [(f[0], g, w) for f, g, w in zip(MatdiffInfo._fields_ + [("eps", 0)], got, want) if not (g == w or (g != g and w != w))])
                n_checked += 1
    assert n_checked > 100
    assert L.libxsmm_matdiff(C.byref(MatdiffInfo()), gen.F64, 4, 4, None, None, None, None) != 0            # no data at all
    for bad in (26, gen.U8):    # UNSUPPORTED, and plain U8 which the reference does not compare either
        assert L.libxsmm_matdiff(C.byref(MatdiffInfo()), bad, 4, 4, a.ctypes.data, a.ctypes.data, None, None) != 0


def test_matdiff_reduce_matches_reference():
    rng = np.random.default_rng(12)
    m, n, count = 17, 9, 5
    a = rng.standard_normal(m * n * count); b = a + rng.standard_normal(m * n * count) * np.repeat(10.0 ** -rng.integers(2, 9, size=count), m * n)

    def run_ref():
        want = np.zeros(27)
        assert ref_lib.ref_matdiff_reduce(gen.F64, m, n, count, a.ctypes.data, b.ctypes.data, want.ctypes.data) == 0
        return want
    want = R.value(run_ref)
    total = MatdiffInfo(); L.libxsmm_matdiff_clear(C.byref(total))
    for i in range(count):
        d = MatdiffInfo()
        assert L.libxsmm_matdiff(C.byref(d), gen.F64, m, n, a[i * m * n:].ctypes.data, b[i * m * n:].ctypes.data, None, None) == 0
        L.libxsmm_matdiff_reduce(C.byref(total), C.byref(d))
    assert _same(_image(total), want)


def test_rng_conversions_and_matinit_match_reference():
    L.libxsmm_rng_set_seed.argtypes = [C.c_uint]; L.libxsmm_rng_f32_seq.argtypes = [_P, _I]
    L.libxsmm_rng_f64.restype = _D; L.libxsmm_rng_u32.restype, L.libxsmm_rng_u32.argtypes = C.c_uint, [C.c_uint]
    for seed in (555, 1, 0, 4242):
        def run_ref():
            f32_r = np.zeros(100, dtype=np.float32); f64_r = np.zeros(50); u_r = np.zeros(50, dtype=np.uint32)
            ref_lib.ref_rng(seed, f32_r.ctypes.data, 100, f64_r.ctypes.data, 50, u_r.ctypes.data, 50, 1000)
            return np.concatenate([f32_r.view(np.uint8), f64_r.view(np.uint8), u_r.view(np.uint8)])
        f32_o = np.zeros(100, dtype=np.float32)
        L.libxsmm_rng_set_seed(seed); L.libxsmm_rng_f32_seq(f32_o.ctypes.data, 100)
        f64_o = np.array([L.libxsmm_rng_f64() for _ in range(50)]); u_o = np.array([L.libxsmm_rng_u32(1000) for _ in range(50)], dtype=np.uint32)
        R.same(run_ref, np.concatenate([f32_o.view(np.uint8), f64_o.view(np.uint8), u_o.view(np.uint8)]), seed)
        assert f32_o.min() >= 0 and f32_o.max() < 1
    # low-precision array conversions, all 8-bit codes and a spread of f32 values incl. specials
    rng = np.random.default_rng(13)
    f = np.concatenate([rng.standard_normal(4000).astype(np.float32) * np.float32(10.0) ** rng.integers(-8, 6, size=4000).astype(np.float32),
                        np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 448.0, 464.0, 465.0, 1e-3, 2 ** -9, 2 ** -10, 1.5 * 2 ** -9, 57344.0, 61440.0, 65504.0, 1e-40],
                                 dtype=np.float32)])
    codes8 = np.arange(256, dtype=np.uint8); codes16 = rng.integers(0, 65536, size=4000).astype(np.uint16)
    names = ["libxsmm_rne_convert_fp32_bf8", "libxsmm_convert_bf8_f32", "libxsmm_rne_convert_fp32_hf8", "libxsmm_convert_hf8_f32", "libxsmm_rne_convert_fp32_bf16",
             "libxsmm_rnaz_convert_fp32_bf16", "libxsmm_truncate_convert_f32_bf16", "libxsmm_convert_bf16_f32", "libxsmm_rne_convert_fp32_f16", "libxsmm_convert_f16_f32"]
    for which, name in enumerate(names):
        src = {1: codes8, 3: codes8, 7: codes16, 9: codes16}.get(which, f)
        odt = np.float32 if which in (1, 3, 7, 9) else (np.uint8 if which in (0, 2) else np.uint16)
        def run_ref():
            want = np.zeros(len(src), dtype=odt)
            ref_lib.ref_lp_convert(which, src.ctypes.data, want.ctypes.data, len(src))
            return want.view(np.uint8)
        got = np.zeros(len(src), dtype=odt)
        fn = getattr(L, name); fn.restype, fn.argtypes = None, [_P, _P, C.c_size_t]
        fn(src.ctypes.data, got.ctypes.data, len(src))
        R.same(run_ref, got.view(np.uint8), name)
    # external generator state (DROPOUT / STOCHASTIC_ROUND callers), stochastic bf8 conversion, 2^x and nearbyint helpers
    L.libxsmm_rng_create_extstate.restype, L.libxsmm_rng_create_extstate.argtypes = C.POINTER(C.c_uint), [C.c_uint]
    L.libxsmm_rng_destroy_extstate.restype, L.libxsmm_rng_destroy_extstate.argtypes = None, [C.POINTER(C.c_uint)]
    L.libxsmm_rng_get_extstate_size.restype = C.c_uint
    assert L.libxsmm_rng_get_extstate_size() == 256
    for seed in (0, 1, 555, 0xfffffff0):
        def run_ref():
            want = np.zeros(64, dtype=np.uint32); ref_lib.ref_extstate(seed, want.ctypes.data)
            return want
        st = L.libxsmm_rng_create_extstate(seed)
        got = np.ctypeslib.as_array(st, shape=(64,)).copy(); L.libxsmm_rng_destroy_extstate(st)
        R.same(run_ref, got, seed)
    L.libxsmm_stochastic_convert_fp32_bf8.restype, L.libxsmm_stochastic_convert_fp32_bf8.argtypes = None, [_P, _P, C.c_uint, _P, C.c_uint]
    for n_, start in ((1, 0), (1, 13), (37, 5), (4016, 0)):
        x = f[:n_].copy()
        s0 = ((np.arange(64, dtype=np.uint64) * 2654435761 + 12345) % (2 ** 32)).astype(np.uint32)

        def run_ref():
            s_r = s0.copy(); o_r = np.zeros(n_, dtype=np.uint8)
            ref_lib.ref_stochastic_bf8(x.ctypes.data, o_r.ctypes.data, n_, s_r.ctypes.data, start)
            return np.concatenate([o_r, s_r.view(np.uint8)])
        s_o = s0.copy(); o_o = np.zeros(n_, dtype=np.uint8)
        L.libxsmm_stochastic_convert_fp32_bf8(x.ctypes.data, o_o.ctypes.data, n_, s_o.ctypes.data, start)
        R.same(run_ref, np.concatenate([o_o, s_o.view(np.uint8)]), (n_, start))
    L.libxsmm_sexp2_i8i.restype, L.libxsmm_sexp2_i8i.argtypes = C.c_float, [_I]
    es = range(-128, 128)
    R.same(lambda: np.array([ref_lib.ref_sexp2_i8i(e) for e in es], dtype=np.float32), np.array([L.libxsmm_sexp2_i8i(e) for e in es], dtype=np.float32), "sexp2")
    L.libxsmm_nearbyintf.restype, L.libxsmm_nearbyintf.argtypes = C.c_float, [C.c_float]
    vs = (0.5, 1.5, 2.5, -0.5, -1.5, 3.49999, 1e9, -7.5000001)
    R.same(lambda: np.array([ref_lib.ref_nearbyintf(v) for v in vs], dtype=np.float32), np.array([L.libxsmm_nearbyintf(v) for v in vs], dtype=np.float32), "nearbyint")
    # coprime2 and the drivers' fill macro (compiled from OUR header)
    L.libxsmm_coprime2.restype, L.libxsmm_coprime2.argtypes = C.c_size_t, [C.c_size_t]
    nns = list(range(0, 300)) + [1000, 4096, 5000, 65536, 99991, 1000000, 128 * 1000000 // 7]
    R.same(lambda: np.array([ref_lib.ref_coprime2(nn) for nn in nns], dtype=np.uint64), np.array([L.libxsmm_coprime2(nn) for nn in nns], dtype=np.uint64), "coprime2")
    so = os.path.join(ROOT, "build", "utils_probe.so")
    os.makedirs(os.path.dirname(so), exist_ok=True)
    subprocess.check_call(["gcc", "-O1", "-shared", "-fPIC", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "utils_probe.c"), "-o", so,
                           "-L" + os.path.join(ROOT, "libxsmm_b200", "lib"), "-lxsmm", "-Wl,-rpath," + os.path.join(ROOT, "libxsmm_b200", "lib")])
    probe = C.CDLL(so)
    assert probe.probe_datatype_double() == gen.F64 and probe.probe_datatype_float() == gen.F32 and probe.probe_flags() == 2 + 1024
    probe.probe_matinit.argtypes = [_I, _D, _P, _I, _I, _I, _D]
    for is64, npdt in ((1, np.float64), (0, np.float32)):
        for (seed, nr, nc, ld, scale) in ((0, 96, 48, 96, 1.0), (0, 13, 7, 16, 0.5), (42, 13, 7, 16, 1.0), (1, 5, 5, 5, 2.0)):
            def run_ref():
                a = np.full(ld * nc, 7, dtype=npdt)
                ref_lib.ref_matinit(is64, float(seed), a.ctypes.data, nr, nc, ld, scale)
                return a
            b = np.full(ld * nc, 7, dtype=npdt)
            probe.probe_matinit(is64, float(seed), b.ctypes.data, nr, nc, ld, scale)
            R.same(run_ref, b, (is64, seed, nr, nc, ld))


def test_timer_and_queries():
    L.libxsmm_timer_tick.restype = C.c_ulonglong
    L.libxsmm_timer_duration.restype, L.libxsmm_timer_duration.argtypes = _D, [C.c_ulonglong, C.c_ulonglong]
    import time
    t0 = L.libxsmm_timer_tick(); time.sleep(0.05); t1 = L.libxsmm_timer_tick()
    assert 0.04 < L.libxsmm_timer_duration(t0, t1) < 0.5 and L.libxsmm_timer_duration(t1, t0) == L.libxsmm_timer_duration(t0, t1)
    L.libxsmm_cpuid_dot_pack_factor.argtypes = [_I]
    assert [L.libxsmm_cpuid_dot_pack_factor(t) for t in (gen.BF16, gen.F16, gen.I8, gen.U8, gen.F32, gen.F64)] == [2, 2, 4, 4, 1, 1]
    L.libxsmm_cpuid.argtypes = [_P]
    assert L.libxsmm_cpuid(None) > 1104           # above LIBXSMM_X86_AVX512_SPR: the drivers' "has bf16/int8 matrix units" test holds
    L.libxsmm_stristr.restype, L.libxsmm_stristr.argtypes = C.c_char_p, [C.c_char_p, C.c_char_p]
    assert L.libxsmm_stristr(b"Target=SPR", b"spr") == b"SPR" and L.libxsmm_stristr(b"abc", b"x") is None
