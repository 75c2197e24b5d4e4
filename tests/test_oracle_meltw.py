"""CPU-only: pins the mateltwise restatement (oracle/oracle_meltw.c) against libxsmm_reference_elementwise of the
UNMODIFIED reference (oracle/_ref) on seeded inputs, bit for bit -- including the transcendental ops, which call the
same libm functions in the same order on the same host. Where the reference is not built, its stored answers stand in
for it (tests/ref_answers.py)."""
import ctypes as C

import numpy as np
import pytest

import gen
import libxsmm_b200 as X     # only for the enumerators and argument structs (no kernel is launched)
import ref_answers as R
from oracle_ffi import iarr, oracle, ref
UNS = gen.F64 + 26


def rnd(rng, n, t, positive=False):
    x = rng.standard_normal(n).astype(np.float32)
    if positive:
        x = np.abs(x) + 0.1
    if t == gen.F32:
        return x
    if t == gen.F64:
        return x.astype(np.float64)
    if t == gen.BF16:
        return gen.f32_to_bf16_bits(x)
    return x.astype(np.float16).view(np.uint16)


def both(desc, make_param, outs):
    """run reference and restatement on identical copies; `outs` lists the output arrays (copied per side)"""
    def run(side):
        bufs = [o.copy() for o in outs]
        keep = []
        p = make_param(bufs, keep)
        rc = side["meltw"](iarr(*desc), C.addressof(p), 0)
        assert rc == 0, (desc, rc)
        return np.concatenate([b.view(np.uint8).ravel() for b in bufs])
    R.same(lambda: run(ref), run(oracle), desc)


UNARY = ["IDENTITY", "XOR", "X2", "SQRT", "NEGATE", "INC", "RECIPROCAL", "RECIPROCAL_SQRT", "TANH", "TANH_INV", "SIGMOID", "SIGMOID_INV", "GELU", "GELU_INV", "EXP"]


@pytest.mark.parametrize("tin,tout", [(gen.F32, gen.F32), (gen.BF16, gen.BF16), (gen.F16, gen.F32), (gen.F32, gen.BF16), (gen.BF16, gen.F16), (gen.F64, gen.F64)])
def test_unary_map_ops(tin, tout):
    rng = np.random.default_rng(61)
    for name in (UNARY[:8] if tin == gen.F64 else UNARY):
        op = getattr(X, "MELTW_TYPE_UNARY_" + name)
        for (m, n, pad, bc) in ((33, 17, 0, 0), (100, 3, 5, 0), (1, 64, 2, 0), (40, 9, 0, X.MELTW_FLAG_UNARY_BCAST_ROW),
                                (40, 9, 0, X.MELTW_FLAG_UNARY_BCAST_COL), (7, 7, 1, X.MELTW_FLAG_UNARY_BCAST_SCALAR)):
            ldi, ldo = m + pad, m + 2 * pad
            x = rnd(rng, ldi * n, tin, positive=name in ("SQRT", "RECIPROCAL", "RECIPROCAL_SQRT")); y0 = rnd(rng, ldo * n, tout)
            tcomp = gen.F64 if tin == gen.F64 else gen.F32

            def mk(bufs, keep):
                p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary = x.ctypes.data, bufs[0].ctypes.data
                return p
            both((1, op, bc, m, n, ldi, 0, 0, ldo, tin, UNS, UNS, tout, tcomp), mk, [y0])


@pytest.mark.parametrize("t", [gen.F32, gen.BF16, gen.F16])
def test_relu_family_and_masks(t):
    rng = np.random.default_rng(62)
    for fwd, inv in (("RELU", "RELU_INV"), ("LEAKY_RELU", "LEAKY_RELU_INV"), ("ELU", "ELU_INV")):
        for (m, n, pad) in ((35, 11, 0), (64, 5, 3), (9, 40, 7)):
            for bitm in ((1, 0) if fwd != "ELU" else (0,)):
                ld = m + pad
                flags = X.MELTW_FLAG_UNARY_BITMASK_2BYTEMULT if bitm else 0
                x = rnd(rng, ld * n, t); y0 = rnd(rng, ld * n, t); alpha = C.c_float(0.3)
                mask0 = rng.integers(0, 256, size=(ld + 15) // 16 * 2 * n, dtype=np.uint8)
                op = getattr(X, "MELTW_TYPE_UNARY_" + fwd)

                def mk(bufs, keep):
                    p = X.MeltwUnaryParam(); p.op.primary = C.addressof(alpha)
                    p.inp.primary, p.out.primary, p.out.secondary = x.ctypes.data, bufs[0].ctypes.data, bufs[1].ctypes.data
                    return p
                both((1, op, flags, m, n, ld, 0, 0, ld, t, UNS, UNS, t, gen.F32), mk, [y0, mask0])
                if fwd == "ELU" or bitm:
                    g = rnd(rng, ld * n, t); o0 = rnd(rng, ld * n, t)
                    aux = rnd(rng, ld * n, t) if fwd == "ELU" else mask0
                    opi = getattr(X, "MELTW_TYPE_UNARY_" + inv)

                    def mki(bufs, keep):
                        p = X.MeltwUnaryParam(); p.op.primary = C.addressof(alpha)
                        p.inp.primary, p.inp.secondary, p.out.primary = g.ctypes.data, aux.ctypes.data, bufs[0].ctypes.data
                        return p
                    both((1, opi, flags, m, n, ld, 0, 0, ld, t, UNS, UNS, t, gen.F32), mki, [o0])


@pytest.mark.parametrize("t", [gen.F32, gen.BF16, gen.F64])
def test_binary_ternary_compare_select(t):
    rng = np.random.default_rng(63)
    tcomp = gen.F64 if t == gen.F64 else gen.F32
    for (m, n, pad) in ((33, 9, 0), (16, 20, 4)):
        ld = m + pad
        a, b, c3, y0 = (rnd(rng, ld * n, t) for _ in range(4))
        for name in ("ADD", "MUL", "SUB", "DIV", "MULADD", "MAX", "MIN"):
            for bc in (0, X.MELTW_FLAG_BINARY_BCAST_COL_IN_0, X.MELTW_FLAG_BINARY_BCAST_ROW_IN_1, X.MELTW_FLAG_BINARY_BCAST_SCALAR_IN_1):
                def mk(bufs, keep):
                    p = X.MeltwBinaryParam(); p.in0.primary, p.in1.primary, p.out.primary = a.ctypes.data, b.ctypes.data, bufs[0].ctypes.data
                    return p
                both((2, getattr(X, "MELTW_TYPE_BINARY_" + name), bc, m, n, ld, ld, 0, ld, t, t, UNS, t, tcomp), mk, [y0])
        if t != gen.F64:
            mask0 = rng.integers(0, 256, size=(ld + 15) // 16 * 2 * n, dtype=np.uint8)
            for name in ("GT", "GE", "LT", "LE", "EQ", "NE"):
                def mkc(bufs, keep):
                    p = X.MeltwBinaryParam(); p.in0.primary, p.in1.primary, p.out.primary = a.ctypes.data, b.ctypes.data, bufs[0].ctypes.data
                    return p
                both((2, getattr(X, "MELTW_TYPE_BINARY_CMP_OP_" + name), X.MELTW_FLAG_BINARY_BITMASK_2BYTEMULT if hasattr(X, "MELTW_FLAG_BINARY_BITMASK_2BYTEMULT") else 0,
                      m, n, ld, ld, 0, ld, t, t, UNS, gen.F32 if False else t, tcomp), mkc, [mask0])
            for name in ("MULADD", "NMULADD"):
                def mkt(bufs, keep):
                    p = X.MeltwTernaryParam(); p.in0.primary, p.in1.primary, p.in2.primary, p.out.primary = a.ctypes.data, b.ctypes.data, c3.ctypes.data, bufs[0].ctypes.data
                    return p
                both((3, getattr(X, "MELTW_TYPE_TERNARY_" + name), 0, m, n, ld, ld, ld, ld, t, t, t, t, tcomp), mkt, [y0])
        sel = rng.integers(0, 256, size=(ld + 15) // 16 * 2 * n, dtype=np.uint8)

        def mks(bufs, keep):
            p = X.MeltwTernaryParam(); p.in0.primary, p.in1.primary, p.in2.primary, p.out.primary = a.ctypes.data, b.ctypes.data, sel.ctypes.data, bufs[0].ctypes.data
            return p
        both((3, X.MELTW_TYPE_TERNARY_SELECT, X.MELTW_FLAG_TERNARY_BITMASK_2BYTEMULT if hasattr(X, "MELTW_FLAG_TERNARY_BITMASK_2BYTEMULT") else 0,
              m, n, ld, ld, ld, ld, t, t, gen.F32 if False else UNS + 0 if False else t, t, tcomp), mks, [y0])


@pytest.mark.parametrize("t", [gen.F32, gen.BF16, gen.F64])
def test_reductions(t):
    rng = np.random.default_rng(64)
    for (m, n, pad) in ((33, 17, 0), (8, 70, 3)):
        ldi = m + pad
        x = rnd(rng, ldi * n, t)
        for name in ("X_OP_ADD", "X2_OP_ADD", "X_X2_OP_ADD", "X_OP_MAX", "X_OP_MIN", "X_OP_ABSMAX"):
            if t == gen.F64 and "X2" in name:
                continue    # the reference's F64 path never stores the sums of squares (it zeroes the plane, :1150-1153 and :1282): not restated
            for rows in (1, 0):
                for init in ((0, 1) if "ADD" in name else (0,)):
                    flags = (X.MELTW_FLAG_UNARY_REDUCE_ROWS if rows else X.MELTW_FLAG_UNARY_REDUCE_COLS) | (X.MELTW_FLAG_UNARY_REDUCE_INIT_ACC if init else 0)
                    ldo = n if rows else m      # ldo > m: the reference also stores its (uninitialised) scratch for rows m..ldo-1 (:1425-1430): not part of the contract
                    y0 = rnd(rng, 2 * max(ldo, n, m) + 8, t)

                    def mk(bufs, keep):
                        p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary = x.ctypes.data, bufs[0].ctypes.data
                        return p
                    both((1, getattr(X, "MELTW_TYPE_UNARY_REDUCE_" + name), flags, m, n, ldi, 0, 0, ldo, t, UNS, UNS, t, gen.F64 if t == gen.F64 else gen.F32), mk, [y0])


def test_layout_transforms_and_dequant():
    """same matrix of transforms as tests/test_meltw_gpu.py, output buffers pre-filled with random bytes so that every byte
    the reference defines (including the zero padding of the VNNI packers) is compared"""
    rng = np.random.default_rng(65)
    for t in (gen.F64, gen.F32, gen.BF16, gen.I8):
        for (m, n, pi, po) in ((33, 17, 0, 0), (64, 64, 2, 5), (1, 9, 0, 0)):
            ldi, ldo = m + pi, n + po
            x = rng.integers(0, 256, size=ldi * n * gen.TS[t], dtype=np.uint8); o0 = rng.integers(0, 256, size=ldo * m * gen.TS[t], dtype=np.uint8)

            def mk(bufs, keep):
                p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary = x.ctypes.data, bufs[0].ctypes.data
                return p
            both((1, X.MELTW_TYPE_UNARY_TRANSFORM_NORM_TO_NORMT, 0, m, n, ldi, 0, 0, ldo, t, UNS, UNS, t, t), mk, [o0])
    for name, t, v in (("NORM_TO_VNNI2", gen.BF16, 2), ("NORM_TO_VNNI4", gen.I8, 4), ("NORM_TO_VNNI4", gen.BF16, 4), ("NORM_TO_VNNI2T", gen.BF16, 2),
                       ("NORM_TO_VNNI4T", gen.BF16, 4), ("VNNI2_TO_VNNI2T", gen.BF16, 2), ("VNNI4_TO_VNNI4T", gen.I8, 4), ("VNNI4_TO_VNNI4T", gen.BF16, 4),
                       ("VNNI2T_TO_NORM", gen.BF16, 2), ("VNNI4T_TO_NORM", gen.BF16, 4), ("VNNI4_TO_NORM", gen.I8, 4)):
        op = getattr(X, "MELTW_TYPE_UNARY_TRANSFORM_" + name)
        for (m, n, pad) in ((32, 16, 0), (64, 8, 4), (8, 64, 0), (40, 12, 8)):
            ldi = m + pad
            ldo = (n if name in ("VNNI2_TO_VNNI2T", "VNNI4_TO_VNNI4T", "NORM_TO_VNNI2T", "NORM_TO_VNNI4T") else
                   (n if name in ("VNNI2T_TO_NORM", "VNNI4T_TO_NORM") else m)) + pad
            x = rng.integers(0, 256, size=(ldi + 8) * (n + 8) * 4 * gen.TS[t], dtype=np.uint8)
            o0 = rng.integers(0, 256, size=(ldo + 8) * (max(m, n) + 8) * 4 * gen.TS[t], dtype=np.uint8)

            def mkv(bufs, keep):
                p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary = x.ctypes.data, bufs[0].ctypes.data
                return p
            both((1, op, 0, m, n, ldi, 0, 0, ldo, t, UNS, UNS, t, t), mkv, [o0])
    for t, npdt in ((gen.I8, np.int8), (gen.I16, np.int16), (gen.I32, np.int32)):
        m, n, ld = 20, 7, 23
        x = rng.integers(-100, 100, size=ld * n).astype(npdt); y0 = np.zeros(ld * n, dtype=np.float32); scf = C.c_float(0.0625)

        def mkd(bufs, keep):
            p = X.MeltwUnaryParam(); p.inp.primary, p.inp.secondary, p.out.primary = x.ctypes.data, C.addressof(scf), bufs[0].ctypes.data
            return p
        both((1, X.MELTW_TYPE_UNARY_DEQUANT, 0, m, n, ld, 0, 0, ld, t, UNS, UNS, gen.F32, gen.F32), mkd, [y0])


def test_gather_scatter_and_quant():
    rng = np.random.default_rng(66)
    for t, npdt in ((gen.F32, np.float32), (gen.BF16, np.uint16), (gen.I8, np.uint8)):
        for idx8 in (0, 1):
            idt = np.uint64 if idx8 else np.uint32
            f8 = X.MELTW_FLAG_UNARY_IDX_SIZE_8BYTES if idx8 else X.MELTW_FLAG_UNARY_IDX_SIZE_4BYTES
            m, n, big = 19, 11, 40
            # gather columns / rows / offsets out of a big x big source
            src = rng.integers(0, 250, size=big * big).astype(npdt)
            for mode, idx in ((X.MELTW_FLAG_UNARY_GS_COLS, rng.integers(0, big, size=n)), (X.MELTW_FLAG_UNARY_GS_ROWS, rng.integers(0, big, size=m)),
                              (X.MELTW_FLAG_UNARY_GS_OFFS, rng.integers(0, big * big, size=m * n))):
                ia = idx.astype(idt); y0 = np.zeros((m + 2) * n, dtype=npdt)

                def mk(bufs, keep):
                    p = X.MeltwUnaryParam(); p.inp.primary, p.inp.secondary, p.out.primary = src.ctypes.data, ia.ctypes.data, bufs[0].ctypes.data
                    return p
                both((1, X.MELTW_TYPE_UNARY_GATHER, mode | f8, m, n, big, 0, 0, m + 2, t, UNS, UNS, t, t), mk, [y0])
            # scatter with unique targets (the result must not depend on the visiting order)
            x = rng.integers(0, 250, size=(m + 1) * n).astype(npdt)
            for mode, idx in ((X.MELTW_FLAG_UNARY_GS_COLS, rng.permutation(big)[:n]), (X.MELTW_FLAG_UNARY_GS_ROWS, rng.permutation(big)[:m]),
                              (X.MELTW_FLAG_UNARY_GS_OFFS, rng.permutation(big * big)[:m * n])):
                ia = idx.astype(idt); y0 = rng.integers(0, 250, size=big * big).astype(npdt)

                def mks(bufs, keep):
                    p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary, p.out.secondary = x.ctypes.data, bufs[0].ctypes.data, ia.ctypes.data
                    return p
                both((1, X.MELTW_TYPE_UNARY_SCATTER, mode | f8, m, n, m + 1, 0, 0, big, t, UNS, UNS, t, t), mks, [y0])
    for tout, npdt in ((gen.I8, np.int8), (gen.I16, np.int16), (gen.I32, np.int32)):
        for sat in (0, X.MELTW_FLAG_UNARY_SIGN_SAT_QUANT):
            m, n, ld = 23, 9, 25
            x = (rng.standard_normal(ld * n) * 90).astype(np.float32); y0 = np.zeros(ld * n, dtype=npdt); scf = C.c_float(1.75)

            def mkq(bufs, keep):
                p = X.MeltwUnaryParam(); p.inp.primary, p.inp.secondary, p.out.primary = x.ctypes.data, C.addressof(scf), bufs[0].ctypes.data
                return p
            both((1, X.MELTW_TYPE_UNARY_QUANT, sat, m, n, ld, 0, 0, ld, gen.F32, UNS, UNS, tout, gen.F32), mkq, [y0])


def test_eight_bit_float_element_types():
    """BF8 (E5M2) and HF8 (E4M3) as input / output element types of the map kernels: every byte pattern as input, f32 values over the
    whole exponent range (incl. halfway cases, overflow, sub-normal results) as output"""
    rng = np.random.default_rng(69)
    m, n, ld = 64, 16, 66
    wide = (rng.standard_normal(ld * n) * np.exp2(rng.integers(-22, 18, size=ld * n))).astype(np.float32)
    wide[::5] = np.ldexp(rng.integers(8, 32, size=wide[::5].size) / 16.0 + 1.0 / 32.0, rng.integers(-12, 10, size=wide[::5].size)).astype(np.float32)   # exact ties
    wide[3] = np.inf; wide[4] = -np.inf; wide[7] = np.nan; wide[9] = 448.0; wide[10] = 464.0; wide[11] = 480.0; wide[12] = 57344.0; wide[13] = 61440.0
    allbytes = np.resize(np.arange(256, dtype=np.uint8), ld * n)
    for t8 in (gen.BF8, gen.HF8):
        for name in ("IDENTITY", "X2", "NEGATE", "RELU"):
            op = getattr(X, "MELTW_TYPE_UNARY_" + name)
            for tin, tout, x in ((gen.F32, t8, wide), (t8, gen.F32, allbytes), (t8, t8, allbytes), (gen.BF16, t8, gen.f32_to_bf16_bits(wide)), (t8, gen.F16, allbytes)):
                y0 = np.zeros(ld * n * (4 if tout == gen.F32 else (2 if tout in (gen.F16, gen.BF16) else 1)), dtype=np.uint8)

                def mk(bufs, keep):
                    p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary = x.ctypes.data, bufs[0].ctypes.data
                    return p
                both((1, op, 0, m, n, ld, 0, 0, ld, tin, UNS, UNS, tout, gen.F32), mk, [y0])
    # binary add with mixed 8-bit inputs
    a8, b8 = rng.integers(0, 256, size=ld * n, dtype=np.uint8), rng.integers(0, 256, size=ld * n, dtype=np.uint8)
    y0 = np.zeros(ld * n, dtype=np.uint8)

    def mkb(bufs, keep):
        p = X.MeltwBinaryParam(); p.in0.primary, p.in1.primary, p.out.primary = a8.ctypes.data, b8.ctypes.data, bufs[0].ctypes.data
        return p
    both((2, X.MELTW_TYPE_BINARY_ADD, 0, m, n, ld, ld, 0, ld, gen.BF8, gen.HF8, UNS, gen.HF8, gen.F32), mkb, [y0])


def test_stochastic_rounding_to_bf8_and_dump():
    """STOCHASTIC_ROUND (unary, binary, ternary) with a BF8 output: bytes AND the advanced 4 x 16-word generator state; DUMP writes twice"""
    rng = np.random.default_rng(72)
    m, n, ld = 37, 13, 40
    x = (rng.standard_normal(ld * n) * np.exp2(rng.integers(-18, 14, size=ld * n))).astype(np.float32)
    x[5] = np.inf; x[6] = np.nan; x[7] = 3.0e-6; x[8] = -1.0e-7
    y = rng.standard_normal(ld * n).astype(np.float32); z = rng.standard_normal(ld * n).astype(np.float32)
    state0 = rng.integers(0, 2 ** 32, size=64, dtype=np.uint32)
    o0 = np.zeros(ld * n, dtype=np.uint8)
    for name in ("IDENTITY", "X2", "DUMP"):
        def mk(bufs, keep):
            p = X.MeltwUnaryParam(); p.op.secondary = bufs[1].ctypes.data
            p.inp.primary, p.out.primary, p.out.secondary = x.ctypes.data, bufs[0].ctypes.data, bufs[2].ctypes.data
            return p
        both((1, getattr(X, "MELTW_TYPE_UNARY_" + name), X.MELTW_FLAG_UNARY_STOCHASTIC_ROUND, m, n, ld, 0, 0, ld, gen.F32, UNS, UNS, gen.BF8, gen.F32), mk, [o0, state0, o0])

    def mkb(bufs, keep):
        p = X.MeltwBinaryParam(); p.op.secondary = bufs[1].ctypes.data
        p.in0.primary, p.in1.primary, p.out.primary = x.ctypes.data, y.ctypes.data, bufs[0].ctypes.data
        return p
    both((2, X.MELTW_TYPE_BINARY_MUL, X.MELTW_FLAG_BINARY_STOCHASTIC_ROUND, m, n, ld, ld, 0, ld, gen.F32, gen.F32, UNS, gen.BF8, gen.F32), mkb, [o0, state0])

    def mkt(bufs, keep):
        p = X.MeltwTernaryParam(); p.op.secondary = bufs[1].ctypes.data
        p.in0.primary, p.in1.primary, p.in2.primary, p.out.primary = x.ctypes.data, y.ctypes.data, z.ctypes.data, bufs[0].ctypes.data
        return p
    both((3, X.MELTW_TYPE_TERNARY_MULADD, X.MELTW_FLAG_TERNARY_STOCHASTIC_ROUND, m, n, ld, ld, ld, ld, gen.F32, gen.F32, gen.F32, gen.BF8, gen.F32), mkt, [o0, state0])
    # DUMP without the flag, f32 -> bf16 (the reference has no F64 DUMP: libxsmm_fp64_unary_compute :116-138 rejects it)
    oo = np.zeros(ld * n, dtype=np.uint16)

    def mkd(bufs, keep):
        p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary, p.out.secondary = x.ctypes.data, bufs[0].ctypes.data, bufs[1].ctypes.data
        return p
    both((1, X.MELTW_TYPE_UNARY_DUMP, 0, m, n, ld, 0, 0, ld, gen.F32, UNS, UNS, gen.BF16, gen.F32), mkd, [oo, oo])


def mx_inputs(rng, m, n, ld):
    """bf16 blocks that reach every branch of the block quantisers: wide exponent range, exact ties of the 4-bit code grid, all-zero
    blocks, blocks with Inf / NaN, sub-normal magnitudes"""
    x = (rng.standard_normal(ld * n) * np.exp2(rng.integers(-20, 20, size=ld * n))).astype(np.float32)
    x[::7] = rng.choice(np.array([0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0, 6.0, -0.75, -2.5], dtype=np.float32), size=x[::7].size) * 4.0
    xb = gen.f32_to_bf16_bits(x).reshape(n, ld)
    xb[0, :32] = 0; xb[1, :32] = 0x8000                       # +0 and -0 blocks
    xb[2, 5] = 0x7f80; xb[3, 20] = 0x7fc1; xb[4, 3] = 0xff80   # +Inf, NaN, -Inf inside a block
    xb[5, :32] = rng.integers(1, 0x7f, size=32)               # bf16 sub-normals
    xb[6, :32] = gen.f32_to_bf16_bits(np.full(32, 3.0e38, dtype=np.float32))
    return xb.reshape(-1).copy()


def test_block_scaled_quantisers():
    """bf16 -> MXFP4 (32-blocks, E8M0 scale), NVFP4 (16-blocks, E4M3 scale), MXBF8 (32-blocks): data and scale bytes"""
    rng = np.random.default_rng(70)
    for tout, blk in ((gen.MXFP4X2, 32), (gen.NVFP4X2, 16), (gen.MXBF8, 32)):
        for (m, n, ldi, ldo) in ((64, 9, 64, 64), (96, 8, 100, 128), (32, 7, 32, 32)):
            x = mx_inputs(rng, m, n, ldi)
            y0 = rng.integers(0, 255, size=ldo * n, dtype=np.uint8); s0 = rng.integers(0, 255, size=(ldo // blk) * n + 8, dtype=np.uint8)

            def mk(bufs, keep):
                p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary, p.out.secondary = x.ctypes.data, bufs[0].ctypes.data, bufs[1].ctypes.data
                return p
            both((1, X.MELTW_TYPE_UNARY_QUANT, 0, m, n, ldi, 0, 0, ldo, gen.BF16, UNS, UNS, tout, gen.F32), mk, [y0, s0])


@pytest.mark.parametrize("t", [gen.F32, gen.BF16, gen.F64])
def test_reductions_to_scalar(t):
    rng = np.random.default_rng(67)
    tcomp = gen.F64 if t == gen.F64 else gen.F32
    m, n, ld = 37, 11, 40
    a, b = rnd(rng, ld * n, t), rnd(rng, ld * n, t)
    y0 = rnd(rng, 4, t)

    def mku(bufs, keep):
        p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary = a.ctypes.data, bufs[0].ctypes.data
        return p
    both((1, X.MELTW_TYPE_UNARY_REDUCE_TO_SCALAR_OP_ADD, 0, m, n, ld, 0, 0, ld, t, UNS, UNS, t, tcomp), mku, [y0])

    def mkb(bufs, keep):
        p = X.MeltwBinaryParam(); p.in0.primary, p.in1.primary, p.out.primary = a.ctypes.data, b.ctypes.data, bufs[0].ctypes.data
        return p
    both((2, X.MELTW_TYPE_BINARY_MUL_AND_REDUCE_TO_SCALAR_OP_ADD, 0, m, n, ld, ld, 0, ld, t, t, UNS, t, tcomp), mkb, [y0])


def test_vnni8_pad_and_vnni4_to_vnni2_transforms():
    """the remaining layout transforms of generator_mateltwise_reference_impl.c:489-531, 581-601, 666-686, 712-786, 806-960;
    output buffers pre-filled with random bytes so that the zero padding the reference writes is compared too"""
    rng = np.random.default_rng(68)
    cases_ = [("NORM_TO_VNNI8", gen.BF16, "m"), ("NORM_TO_VNNI8", gen.I8, "m"), ("NORM_TO_VNNI8_PAD", gen.BF16, "m"), ("NORM_TO_VNNI8T", gen.BF16, "n"),
              ("VNNI8_TO_VNNI8T", gen.BF16, "n"), ("VNNI8_TO_VNNI8T", gen.I8, "n"), ("VNNI8T_TO_NORM", gen.BF16, "n"), ("VNNI4_TO_VNNI2", gen.I8, "m"),
              ("PADM_MOD2", gen.BF16, "m"), ("PADN_MOD2", gen.BF16, "m"), ("PADNM_MOD2", gen.BF16, "m"),
              ("PADM_MOD4", gen.I8, "m"), ("PADN_MOD4", gen.I8, "m"), ("PADNM_MOD4", gen.I8, "m")]
    for name, t, ld_of in cases_:
        op = getattr(X, "MELTW_TYPE_UNARY_TRANSFORM_" + name)
        shapes = ((32, 16, 0), (64, 8, 8), (8, 64, 0), (40, 24, 8))
        if name.startswith("PAD") or name == "VNNI4_TO_VNNI2":
            shapes = shapes + ((33, 7, 3), (5, 9, 1)) if name.startswith("PAD") else shapes + ((36, 12, 4),)
        for (m, n, pad) in shapes:
            ldi = m + pad
            ldo = (n if ld_of == "n" else m) + pad
            x = rng.integers(0, 256, size=(ldi + 8) * (n + 16) * 8 * gen.TS[t], dtype=np.uint8)
            o0 = rng.integers(0, 256, size=(ldo + 8) * (max(m, n) + 16) * 8 * gen.TS[t], dtype=np.uint8)

            def mkv(bufs, keep):
                p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary = x.ctypes.data, bufs[0].ctypes.data
                return p
            both((1, op, 0, m, n, ldi, 0, 0, ldo, t, UNS, UNS, t, t), mkv, [o0])


def rng_state(seed):
    """64 words like libxsmm_rng_create_extstate would hand out (any non-degenerate state pins the step function)"""
    return np.random.default_rng(seed).integers(1, 2**32 - 1, size=64, dtype=np.uint64).astype(np.uint32)


@pytest.mark.parametrize("tin,tout", [(gen.F32, gen.F32), (gen.BF16, gen.BF16), (gen.F32, gen.BF16), (gen.F16, gen.F16)])
def test_dropout_forward_and_backward(tin, tout):
    rng = np.random.default_rng(69)
    for (m, n, pad) in ((33, 7, 0), (64, 5, 3), (16, 16, 0), (100, 3, 4), (7, 9, 1)):
        for bitm in (0, X.MELTW_FLAG_UNARY_BITMASK_2BYTEMULT):
            ldi, ldo = m + pad, m + 2 * pad
            x = rnd(rng, ldi * n, tin); y0 = rnd(rng, ldo * n, tout)
            prob = C.c_float(0.3)
            mask0 = rng.integers(0, 256, size=((ldo + 15) // 16 * 16) // 8 * n + 8, dtype=np.uint8)
            st0 = rng_state(m * 131 + n)

            def mk(bufs, keep):
                p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary, p.out.secondary = x.ctypes.data, bufs[0].ctypes.data, bufs[1].ctypes.data
                p.op.primary, p.op.secondary = C.addressof(prob), bufs[2].ctypes.data
                return p
            both((1, X.MELTW_TYPE_UNARY_DROPOUT, bitm, m, n, ldi, 0, 0, ldo, tin, UNS, UNS, tout, gen.F32), mk, [y0, mask0, st0])
            if bitm:
                # backward from a mask laid out against ldi
                maskb = rng.integers(0, 256, size=((ldi + 15) // 16 * 16) // 8 * n + 8, dtype=np.uint8)

                def mkb(bufs, keep):
                    p = X.MeltwUnaryParam(); p.inp.primary, p.inp.secondary, p.out.primary = x.ctypes.data, maskb.ctypes.data, bufs[0].ctypes.data
                    p.op.primary = C.addressof(prob)
                    return p
                both((1, X.MELTW_TYPE_UNARY_DROPOUT_INV, bitm, m, n, ldi, 0, 0, ldo, tin, UNS, UNS, tout, gen.F32), mkb, [y0])


def test_unzip_and_decompose_to_bf16_planes():
    rng = np.random.default_rng(70)
    for (m, n, pad) in ((33, 7, 0), (64, 5, 3), (1, 9, 2)):
        ldi, ldo = m + pad, m + 2 * pad
        x = (rng.standard_normal(ldi * n) * np.exp(rng.uniform(-8, 8, ldi * n))).astype(np.float32)
        plane = ldo * n + 5
        for name, nplanes in (("UNZIP", 2), ("DECOMP_FP32_TO_BF16X2", 2), ("DECOMP_FP32_TO_BF16X3", 3)):
            o0 = rng.integers(0, 60000, size=plane * nplanes, dtype=np.uint16)
            offs = np.array([plane * 2, plane * 4], dtype=np.uint64)

            def mk(bufs, keep):
                p = X.MeltwUnaryParam(); p.inp.primary, p.out.primary, p.out.secondary = x.ctypes.data, bufs[0].ctypes.data, offs.ctypes.data
                return p
            both((1, getattr(X, "MELTW_TYPE_UNARY_" + name), 0, m, n, ldi, 0, 0, ldo, gen.F32, UNS, UNS, gen.BF16, gen.F32), mk, [o0])
