"""CPU-only: pins oracle/oracle.c (the restatement) against the UNMODIFIED reference (oracle/_ref/libxsmm_ref.so)
on seeded inputs -- bit for bit -- and against the reference's JIT path (AMX/AVX-512) within the reference's own
acceptance norms. Where the reference is not built, its stored answers stand in for it (tests/ref_answers.py)."""
import ctypes as C

import numpy as np
import pytest

import cases
import gen
import ref_answers as R
from oracle_ffi import iarr, oracle, ref, run_gemm


def test_conversions_match_reference():
    rng = np.random.default_rng(1)
    bits = np.concatenate([rng.integers(0, 2**32, size=20000, dtype=np.uint64).astype(np.uint32),
                           np.array([0, 0x80000000, 0x7f800000, 0xff800000, 0x7fc00000, 0x7f800001, 0x00000001, 0x007fffff,
                                     0x38800000, 0x387fffff, 0x33000000, 0x33000001, 0x477fe000, 0x477ff000, 0x47800000], dtype=np.uint32)])
    fs = [float(f) for f in bits.view(np.float32)]
    for name in ("f32_to_bf16", "f32_to_f16"):
        R.same(lambda: np.array([ref[name](f) for f in fs], dtype=np.uint16), np.array([oracle[name](f) for f in fs], dtype=np.uint16), name)
    for name in ("f16_to_f32", "bf16_to_f32"):      # NaN == NaN whatever the payload
        R.same(lambda: np.array([ref[name](h) for h in range(0, 65536, 7)], dtype=np.float32),
               np.array([oracle[name](h) for h in range(0, 65536, 7)], dtype=np.float32), name)


def test_gemm_restatement_is_bit_exact():
    n = 0
    for case in cases.small_cases():
        ops = cases.Operands(case, seed=555 + n)
        got = cases.ref_result(oracle, case, ops, run_gemm)
        R.same(lambda: cases.ref_result(ref, case, ops, run_gemm).view(np.uint8), got.view(np.uint8), case)
        n += 1
    assert n > 300


def test_reference_jit_agrees_with_reference_kernel():
    """the JIT'ed x86 kernels (the CPU baseline) against the C kernel, reference thresholds (gemm_kernel.c:5312-5414);
    the C kernel's answer is the restatement's (bit for bit, test_gemm_restatement_is_bit_exact)"""
    for t, thr in (((gen.F32, gen.F32, gen.F32, gen.F32), 1.2e-5), ((gen.BF16, gen.BF16, gen.F32, gen.F32), 1.2e-5),
                   ((gen.BF16, gen.BF16, gen.F32, gen.BF16), 5e-3), ((gen.U8, gen.I8, gen.I32, gen.I32), 0.0)):
        flags = cases.FLAG_BETA_0 | (cases.FLAG_VNNI_A if t[0] != gen.F32 else 0)
        case = cases.GemmCase(64, 64, 64, *t, flags=flags, br_type=3, br=8)
        ops = cases.Operands(case)
        c_ref = ops.c0.copy()
        assert run_gemm(oracle, case.dims, case.types, case.flags, 3, ops.stride_a, ops.stride_b, 8, ops.a, ops.b, c_ref, mode=0) == 0

        def jit():
            c_jit = ops.c0.copy()
            rc = run_gemm(ref, case.dims, case.types, case.flags, 3, ops.stride_a, ops.stride_b, 8, ops.a, ops.b, c_jit, mode=1)
            assert rc in (0, 2)
            return gen.to_f64(c_jit, t[3])
        c_jit, c_ref = R.sampled(jit, gen.to_f64(c_ref, t[3]))
        assert gen.normf_rel(c_ref, c_jit) <= thr


def _bcsc_inputs(rng, ta, tb, tc, mblocks, M, K, N, bk, bn, density, vnni_a=True, trans_a=False):
    nbr, nbc = K // bk, N // bn
    keep = rng.random((nbc, nbr)) < density
    colptr = np.zeros(nbc + 1, dtype=np.uint32); rowidx = []
    for j in range(nbc):
        rows = np.nonzero(keep[j])[0]
        rowidx.extend(rows.tolist()); colptr[j + 1] = len(rowidx)
    rowidx = np.array(rowidx if rowidx else [0], dtype=np.uint32)
    nnzb = int(colptr[-1])
    bvals = gen.values(rng, max(nnzb, 1) * bk * bn, tb)
    a = gen.values(rng, mblocks * K * M, ta)
    c0 = gen.values(rng, mblocks * N * M, tc)
    return a, bvals, colptr, rowidx, c0


def _run_bcsc(side, types, geo, flags, a, bvals, colptr, rowidx, c):
    from oracle_ffi import iarr
    return side["bcsc"](iarr(*types), iarr(*geo), flags, a.ctypes.data, bvals.ctypes.data, colptr.ctypes.data, rowidx.ctypes.data, c.ctypes.data)


def test_bcsc_oracle_matches_reference_jit():
    """no portable C kernel exists for BCSC in the reference (no fallback for this build kind): the x86 JIT is
    the second opinion; f32 and bf16 accumulate in a different order, integer paths must agree exactly."""
    rng = np.random.default_rng(3)
    for (ta, tb, tcomp, tc), thr in (((gen.F32, gen.F32, gen.F32, gen.F32), 1e-4), ((gen.BF16, gen.BF16, gen.F32, gen.BF16), 5e-3),
                                      ((gen.U8, gen.I8, gen.I32, gen.I32), 0.0), ((gen.I8, gen.U8, gen.I32, gen.I32), 0.0)):
        for beta0 in (1, 0):
            mblocks, M, K, N, bk, bn = 3, 32, 128, 64, 32 if ta != gen.F32 else 16, 16
            flags = (cases.FLAG_BETA_0 if beta0 else 0) | (cases.FLAG_VNNI_A if ta != gen.F32 else 0)
            a, bvals, colptr, rowidx, c0 = _bcsc_inputs(rng, ta, tb, tc, mblocks, M, K, N, bk, bn, 0.5)
            geo = (mblocks, M, K, N, bk, bn)
            c_o = c0.copy()
            assert _run_bcsc(oracle, (ta, tb, tcomp, tc), geo, flags, a, bvals, colptr, rowidx, c_o) == 0

            def jit():
                c_r = c0.copy()
                return gen.to_f64(c_r, tc) if _run_bcsc(ref, (ta, tb, tcomp, tc), geo, flags, a, bvals, colptr, rowidx, c_r) == 0 else None
            c_r, c_o = R.sampled(jit, gen.to_f64(c_o, tc))
            if c_r is None:
                pytest.skip("reference JIT cannot build BCSC for this host ISA")
            err = gen.normf_rel(c_r, c_o)
            assert err <= thr, ((ta, tb, tc), beta0, err)


def test_fsspmdm_oracle_matches_reference():
    rng = np.random.default_rng(4)
    for dtype, eps in ((gen.F32, 1e-4), (gen.F64, 1e-8)):
        for beta in (0.0, 1.0):
            M, K, N = 24, 40, 96
            npdt = gen.NP_OF[dtype]
            a = (gen.values(rng, M * K, gen.F64) * (rng.random(M * K) < 0.2)).astype(npdt)
            b = gen.values(rng, K * N, dtype); c0 = gen.values(rng, M * N, dtype)
            alpha = np.array([1.5], dtype=npdt); bt = np.array([beta], dtype=npdt)
            c_o = c0.copy()
            args = (dtype, M, N, K, K, N, N, alpha.ctypes.data, bt.ctypes.data, a.ctypes.data, b.ctypes.data)
            assert oracle["fsspmdm"](*args, c_o.ctypes.data) == 0

            def run_ref():
                c_r = c0.copy()
                assert ref["fsspmdm"](*args, c_r.ctypes.data) == 0
                return c_r
            c_r, c_o = R.sampled(run_ref, c_o)
            assert gen.normf_rel(c_r, c_o) <= eps
    # invalid inputs answer "no handle" on both sides (N not a multiple of the vector length, beta=2, empty A)
    M, K, N = 8, 8, 24
    a = np.ones(M * K, dtype=np.float32); b = np.ones(K * N, dtype=np.float32); c = np.zeros(M * N, dtype=np.float32)
    one = np.array([1.0], dtype=np.float32); two = np.array([2.0], dtype=np.float32)
    z = np.zeros(M * K, dtype=np.float32)

    def rcs(side):
        return np.array([side["fsspmdm"](gen.F32, M, N, K, K, N, N, one.ctypes.data, one.ctypes.data, a.ctypes.data, b.ctypes.data, c.ctypes.data),
                         side["fsspmdm"](gen.F32, M, 32, K, K, 32, 32, one.ctypes.data, two.ctypes.data, a.ctypes.data, b.ctypes.data, c.ctypes.data),
                         side["fsspmdm"](gen.F32, M, 32, K, K, 32, 32, one.ctypes.data, one.ctypes.data, z.ctypes.data, b.ctypes.data, c.ctypes.data)])
    assert np.all(rcs(oracle) != 0) and np.all(R.value(lambda: rcs(ref)) != 0)


@pytest.mark.parametrize("kind", ["a_csr", "b_csr", "b_csc", "c_csc"])
def test_packed_sparse_oracle_matches_reference_jit(kind):
    """oracle_packed_sp (restated driver golds, samples/xgemm_norm_packed/*.c) against the reference's own JIT of
    libxsmm_create_packed_spgemm_csr/_csc (src/libxsmm_main.c:3553-3638) -- EDGE sizes, f32/f64, beta 0/1."""
    rng = np.random.default_rng(77)
    ran = 0
    for dtype, eps in ((gen.F32, 2e-6), (gen.F64, 1e-14)):
        for (M, N, K, P) in ((9, 9, 9, 8), (20, 9, 35, 16), (56, 9, 56, 64), (35, 20, 9, 16)):
            for beta0 in (0, 1):
                is_csc, dims, ptr, idx, a, b, c0 = cases.packed_sp_case(rng, kind, dtype, M, N, K, P)
                flags = cases.FLAG_BETA_0 if beta0 else 0
                vals = a if kind == "a_csr" else b if kind.startswith("b_") else c0
                c_o = c0.copy()
                args = (is_csc, dtype, iarr(*dims), flags, P, ptr.ctypes.data, idx.ctypes.data, vals.ctypes.data, a.ctypes.data, b.ctypes.data)
                rc_o = oracle["packed_sp"](*args, c_o.ctypes.data)
                if kind == "c_csc" and (dtype != gen.F32 or P % 16):
                    assert rc_o != 0          # C-sparse exists for f32 and whole 16-lane vectors only
                    continue
                assert rc_o == 0
                if kind == "c_csc" and beta0:
                    continue          # reference defect: with BETA_0 the 16-accumulator path stores zmm1 while the sums sit in
                                      # zmm0 (..._csc_csparse_avx_avx2_avx512.c:567-590); the oracle overwrites as documented

                def jit():
                    c_r = c0.copy()
                    return c_r if ref["packed_sp"](*args, c_r.ctypes.data) == 0 else None
                c_r, c_o = R.sampled(jit, c_o)
                if c_r is None:
                    continue          # the JIT declines this (kind, precision, width) on this host
                ran += 1
                assert gen.normf_rel(c_r, c_o) <= eps, (kind, dtype, (M, N, K, P), beta0)
    assert ran > 0, "the reference JIT built none of the cases"


@pytest.mark.parametrize("types", [(gen.F32, gen.F32, gen.F32, gen.F32), (gen.BF16, gen.BF16, gen.F32, gen.BF16), (gen.BF16, gen.BF16, gen.F32, gen.F32),
                                   (gen.F16, gen.F16, gen.F32, gen.F16)])
def test_fused_gemm_restatement_matches_reference(types):
    """oracle_gemm_ext against libxsmm_reference_gemm on the extended ABI: column-bias pre-op, ReLU (+bitmask) / sigmoid post-op,
    VNNI-packed C (generator_gemm_reference_impl.c:255-372, 2803-2842) -- bit for bit (same libm on the same host)"""
    rng = np.random.default_rng(88)
    ta, tb, tcomp, tc = types
    for (m, n, k, pad) in ((32, 16, 32, 0), (13, 6, 8, 3), (64, 64, 64, 0)):
        for beta0 in (1, 0):
            for br_type, br in ((0, 1), (3, 3)):
                for fuse in cases.fused_variants():
                    if fuse[3] and (tc == gen.F32 or n % 2):
                        continue
                    flags = (cases.FLAG_BETA_0 if beta0 else 0) | (cases.FLAG_VNNI_A if ta != gen.F32 and k % 2 == 0 and m % 2 == 0 else 0)
                    case = cases.GemmCase(m, n, k, ta, tb, tcomp, tc, flags=flags, br_type=br_type, br=br, pad=pad)
                    ops = cases.Operands(case, seed=int(rng.integers(1 << 30)))
                    bias = gen.values(rng, m, tc)
                    mask0 = rng.integers(0, 256, size=((case.ldc + 15) // 16 * 16) // 8 * n + 8, dtype=np.uint8)

                    def run(side):
                        c = ops.c0.copy(); mk = mask0.copy()
                        assert cases.run_gemm_ext(side, case, ops, fuse, bias if fuse[0] else None, mk if fuse[2] else None, c) == 0, (case, fuse)
                        return np.concatenate([c.view(np.uint8), mk])      # C, then the mask
                    R.same(lambda: run(ref), run(oracle), (case, fuse))


I4X2 = 18
FLAG_COL_VEC_ZPT, FLAG_INTLV_A, FLAG_BITMASK_A, FLAG_MXK_ZPT = 131072, 262144, 524288, 1048576


def int4_case(rng, m, n, k, br, pad=0):
    lda, ldb, ldc = m + pad, k + pad, m + pad
    blk_a, blk_b = (k // 8) * lda * 4, n * ldb
    a = rng.integers(0, 256, size=blk_a * br, dtype=np.uint8)
    b = rng.integers(0, 256, size=blk_b * br, dtype=np.uint8)
    zpt = rng.integers(0, 16, size=max(m, (blk_a * 2 // k) * br + m), dtype=np.uint8)
    c0 = rng.integers(-1000, 1000, size=n * ldc).astype(np.int32)
    return (m, n, k, lda, ldb, ldc), a, b, zpt, c0, blk_a, blk_b


def test_int4_gemm_restatement_is_bit_exact():
    """U4 x U8 -> I32 with zero points (reference :1273-1321): plain and stride batch-reduce, beta 0/1"""
    rng = np.random.default_rng(90)
    for (m, n, k, pad) in ((32, 16, 32, 0), (13, 6, 8, 3), (64, 64, 64, 0), (5, 3, 16, 1)):
        for br_type, br in ((0, 1), (3, 4)):
            for beta0 in (0, 1):
                dims, a, b, zpt, c0, blk_a, blk_b = int4_case(rng, m, n, k, br, pad)
                flags = (cases.FLAG_BETA_0 if beta0 else 0) | cases.FLAG_VNNI_A | FLAG_INTLV_A | (FLAG_MXK_ZPT if br_type else FLAG_COL_VEC_ZPT)
                c_o = c0.copy()
                assert oracle["gemm_i4"](iarr(*dims), flags, br_type, blk_a, blk_b, br, a.ctypes.data, b.ctypes.data, c_o.ctypes.data, zpt.ctypes.data) == 0

                def run_ref():
                    c_r = c0.copy()
                    assert ref["gemm_aux"](iarr(*dims), iarr(I4X2, gen.U8, gen.I32, gen.I32), flags, br_type, blk_a, blk_b, br, a.ctypes.data, b.ctypes.data,
                                           c_r.ctypes.data, 1, zpt.ctypes.data) == 0
                    return c_r
                R.same(run_ref, c_o, (dims, br_type, beta0))


def bitmap_case(rng, m, n, k, ta, tb, tc, density=0.4, pad=0):
    kb = 1 if ta == gen.F32 else 2
    ldb, ldc = k + pad, m + pad
    bits = rng.random((k // kb) * m * kb) < density
    bitmap = np.packbits(bits, bitorder="little")
    bitmap = np.concatenate([bitmap, np.zeros(8, dtype=np.uint8)])
    a = gen.values(rng, int(bits.sum()) + 4, ta)
    b = gen.values(rng, n * ldb, tb); c0 = gen.values(rng, n * ldc, tc)
    return (m, n, k, m, ldb, ldc), a, b, bitmap, c0


def test_bitmap_sparse_a_restatement_is_bit_exact():
    """bitmap-compressed A (DECOMPRESS_A_VIA_BITMASK, reference :857-948): F32 and 16-bit operands, beta 0/1"""
    rng = np.random.default_rng(91)
    for ta, tb, tc in ((gen.F32, gen.F32, gen.F32), (gen.BF16, gen.BF16, gen.F32), (gen.BF16, gen.BF16, gen.BF16), (gen.F16, gen.F16, gen.F16)):
        for (m, n, k, pad) in ((32, 16, 32, 0), (16, 6, 8, 3), (64, 64, 64, 0)):
            for beta0 in (0, 1):
                dims, a, b, bitmap, c0 = bitmap_case(rng, m, n, k, ta, tb, tc, pad=pad)
                flags = (cases.FLAG_BETA_0 if beta0 else 0) | FLAG_BITMASK_A | (cases.FLAG_VNNI_A if ta != gen.F32 else 0)
                c_o = c0.copy()
                assert oracle["gemm_bitmap"](iarr(*dims), iarr(ta, tb, gen.F32, tc), flags, a.ctypes.data, b.ctypes.data, c_o.ctypes.data, bitmap.ctypes.data) == 0

                def run_ref():
                    c_r = c0.copy()
                    assert ref["gemm_aux"](iarr(*dims), iarr(ta, tb, gen.F32, tc), flags, 0, 0, 0, 1, a.ctypes.data, b.ctypes.data, c_r.ctypes.data, 2,
                                           bitmap.ctypes.data) == 0
                    return c_r.view(np.uint8)
                R.same(run_ref, c_o.view(np.uint8), (dims, (ta, tb, tc), beta0))


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_packed_dense_oracle_matches_reference_jit(kind):
    """libxsmm_create_packed_gemm / _ac_rm / _bc_rm (include/libxsmm.h:195-214): restated driver golds against the reference JIT"""
    rng = np.random.default_rng(94)
    ran = 0
    for dtype, eps in ((gen.F32, 3e-6), (gen.F64, 1e-14)):
        for (M, N, K, P, pad) in ((9, 9, 9, 8, 0), (20, 9, 35, 16, 0), (56, 9, 56, 16, 0), (4, 3, 5, 8, 0), (16, 16, 16, 8, 0)):
            if dtype == gen.F32 and P == 8:
                P = 16
            for beta0 in (0, 1):
                dims, a, b, c0 = cases.packed_dense_case(rng, kind, dtype, M, N, K, P, pad)
                flags = cases.FLAG_BETA_0 if beta0 else 0
                c_o = c0.copy()
                assert oracle["packed_dense"](kind, dtype, iarr(*dims), flags, P, a.ctypes.data, b.ctypes.data, c_o.ctypes.data) == 0

                def jit():
                    c_r = c0.copy()
                    return c_r if ref["packed_dense"](kind, dtype, iarr(*dims), flags, P, a.ctypes.data, b.ctypes.data, c_r.ctypes.data) == 0 else None
                c_r, c_o = R.sampled(jit, c_o)
                if c_r is None:
                    continue
                ran += 1
                assert gen.normf_rel(c_r, c_o) <= eps, (kind, dtype, dims, P, beta0)
    assert ran > 0, "the reference JIT built none of the cases"
