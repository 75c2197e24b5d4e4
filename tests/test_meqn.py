"""Matrix equations (libxsmm_meqn_*, reference include/libxsmm.h:149-162) and the user registry (libxsmm_xregister, :106-125).
CPU: tree construction rules and the registry. GPU: whole equations (the patterns of samples/equation/*: elementwise chains with
broadcasts, layernorm/softmax-style reductions) against the reference's own meqn JIT (oracle/_ref, or its stored answers where
the reference is not built: tests/ref_answers.py) on the same inputs."""
import ctypes as C

import numpy as np
import pytest

import gen
import libxsmm_b200 as X
import ref_answers as R
from oracle_ffi import iarr, ref

SING = (0, 0, 0, 0)     # singular argument attributes
F32 = gen.F32


def build(nodes):
    """nodes in pre-order: ('arg', pos, m, n, ld, dtype) | ('u'|'b'|'t', op, dtype, flags); returns the equation index"""
    eq = X.libxsmm_meqn_create()
    assert eq >= 0
    for nd in nodes:
        if nd[0] == "arg":
            rc = X.libxsmm_meqn_push_back_arg(X.libxsmm_create_meqn_arg_metadata(eq, nd[1]), X.libxsmm_create_meqn_arg_shape(nd[2], nd[3], nd[4], nd[5]),
                                              X.libxsmm_create_matrix_arg_attributes(*SING))
        else:
            fn = {"u": X.libxsmm_meqn_push_back_unary_op, "b": X.libxsmm_meqn_push_back_binary_op, "t": X.libxsmm_meqn_push_back_ternary_op}[nd[0]]
            rc = fn(X.libxsmm_create_meqn_op_metadata(eq, -1), nd[1], nd[2], nd[3])
        assert rc == 0, nd
    return eq


def flat(nodes):
    code = {"arg": 1, "u": 2, "b": 3, "t": 4}
    out = []
    for nd in nodes:
        out += [1, 0, nd[5], 0, nd[1], nd[2], nd[3], nd[4]] if nd[0] == "arg" else [code[nd[0]], nd[1], nd[2], nd[3], -1, 0, 0, 0]
    return out


def test_user_registry_roundtrip():
    key = np.frombuffer(b"libxsmm_b200 key #1" + bytes(13), dtype=np.uint8).copy()
    val = np.arange(10, dtype=np.float64)
    assert not X.libxsmm_xdispatch(key.ctypes.data, key.size)
    p = X.libxsmm_xregister(key.ctypes.data, key.size, val.nbytes, val.ctypes.data)
    assert p
    q = X.libxsmm_xdispatch(key.ctypes.data, key.size)
    assert q == p and np.array_equal(np.ctypeslib.as_array(C.cast(q, C.POINTER(C.c_double)), (10,)), val)
    key2 = key.copy(); key2[0] ^= 1
    assert not X.libxsmm_xdispatch(key2.ctypes.data, key2.size)
    assert not X.libxsmm_xregister(key.ctypes.data, 200, 8, None)          # key longer than LIBXSMM_DESCRIPTOR_MAXSIZE
    X.libxsmm_xrelease(key.ctypes.data, key.size)
    assert not X.libxsmm_xdispatch(key.ctypes.data, key.size)


def test_user_registry_enumeration_survives_release():
    """libxsmm_get_registry_begin / _next over LIBXSMM_KERNEL_KIND_USER (reference include/libxsmm.h:105-108); the walk of
    tests/registry.c:133-137 releases each entry and then asks for the successor of the entry it just released"""
    USER = 3
    keys = [np.frombuffer(bytes([7, i]) + bytes(10), dtype=np.uint8).copy() for i in range(5)]
    vals = [np.full(4, 10 + i, dtype=np.int32) for i in range(5)]
    for k, v in zip(keys, vals):
        assert X.libxsmm_xregister(k.ctypes.data, k.size, v.nbytes, v.ctypes.data)
    seen = {}
    kp = C.c_void_p()
    e = X.libxsmm_get_registry_begin(USER, C.byref(kp))
    while e:
        key = bytes(np.ctypeslib.as_array(C.cast(kp.value, C.POINTER(C.c_ubyte)), (12,)))
        if key[0] == 7:
            seen[key[1]] = int(np.ctypeslib.as_array(C.cast(e, C.POINTER(C.c_int)), (4,))[0])
        info = X.KernelInfo()
        assert X.libxsmm_get_kernel_info(e, C.byref(info)) == 0 and info.kind == USER
        e = X.libxsmm_get_registry_next(e, C.byref(kp))
    assert seen == {i: 10 + i for i in range(5)}
    e = X.libxsmm_get_registry_begin(USER, None); n = 0
    while e:
        X.libxsmm_release_kernel(e); n += 1
        e = X.libxsmm_get_registry_next(e, None)
    assert n >= 5 and not X.libxsmm_get_registry_begin(USER, None)
    assert all(not X.libxsmm_xdispatch(k.ctypes.data, k.size) for k in keys)
    big = np.arange(64, dtype=np.int32)          # a released key comes back with a larger payload
    p = X.libxsmm_xregister(keys[0].ctypes.data, keys[0].size, big.nbytes, big.ctypes.data)
    assert p and np.array_equal(np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_int)), (64,)), big)
    X.libxsmm_xrelease(keys[0].ctypes.data, keys[0].size)


def test_tree_construction_is_preorder_and_bounded():
    eq = X.libxsmm_meqn_create()
    meta = X.libxsmm_create_meqn_op_metadata(eq, -1)
    assert X.libxsmm_meqn_push_back_binary_op(meta, X.MELTW_TYPE_BINARY_ADD, F32, 0) == 0
    a = X.libxsmm_create_meqn_arg_shape(8, 4, 8, F32)
    attr = X.libxsmm_create_matrix_arg_attributes(*SING)
    assert X.libxsmm_meqn_push_back_arg(X.libxsmm_create_meqn_arg_metadata(eq, 0), a, attr) == 0
    assert X.libxsmm_meqn_push_back_arg(X.libxsmm_create_meqn_arg_metadata(eq, 1), a, attr) == 0
    assert X.libxsmm_meqn_push_back_arg(X.libxsmm_create_meqn_arg_metadata(eq, 2), a, attr) != 0     # the tree is complete
    assert X.libxsmm_meqn_push_back_arg(X.libxsmm_create_meqn_arg_metadata(12345, 0), a, attr) != 0  # no such equation


EQUATIONS = {
    # out = tanh(a + b) * c
    "chain": lambda m, n: ([("b", X.MELTW_TYPE_BINARY_MUL, F32, 0), ("u", X.MELTW_TYPE_UNARY_TANH, F32, 0), ("b", X.MELTW_TYPE_BINARY_ADD, F32, 0),
                            ("arg", 0, m, n, m, F32), ("arg", 1, m, n, m, F32), ("arg", 2, m, n, m, F32)], [(m, n)] * 3, (m, n)),
    # out = relu(a * colvec + rowbias)   (broadcast column on in1 of the MUL, broadcast row on in1 of the ADD)
    "bcast": lambda m, n: ([("u", X.MELTW_TYPE_UNARY_RELU, F32, 0), ("b", X.MELTW_TYPE_BINARY_ADD, F32, X.MELTW_FLAG_BINARY_BCAST_ROW_IN_1),
                            ("b", X.MELTW_TYPE_BINARY_MUL, F32, X.MELTW_FLAG_BINARY_BCAST_COL_IN_1), ("arg", 0, m, n, m, F32), ("arg", 1, m, 1, m, F32),
                            ("arg", 2, 1, n, 1, F32)], [(m, n), (m, 1), (1, n)], (m, n)),
    # out[i] = sum_j (a[i][j]^2)      (column reduction of a squared matrix: the layernorm building block)
    "reduce": lambda m, n: ([("u", X.MELTW_TYPE_UNARY_REDUCE_X_OP_ADD, F32, X.MELTW_FLAG_UNARY_REDUCE_COLS), ("u", X.MELTW_TYPE_UNARY_X2, F32, 0),
                             ("arg", 0, m, n, m, F32)], [(m, n)], (m, 1)),
    # out = a - exp(b) * c  (ternary NMULADD: in1 - in0*in2)
    "ternary": lambda m, n: ([("t", X.MELTW_TYPE_TERNARY_NMULADD, F32, 0), ("u", X.MELTW_TYPE_UNARY_EXP, F32, 0), ("arg", 1, m, n, m, F32),
                              ("arg", 0, m, n, m, F32), ("arg", 2, m, n, m, F32)], [(m, n)] * 3, (m, n)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(EQUATIONS))
def test_equations_match_the_reference(name):
    import torch  # noqa: F401
    from gpu_util import dev, host
    rng = np.random.default_rng(96)
    for (m, n) in ((32, 16), (13, 7), (100, 33)):
        nodes, in_shapes, (om, on) = EQUATIONS[name](m, n)
        ins = [(rng.standard_normal(a * b) * 0.5).astype(np.float32) for (a, b) in in_shapes]

        def run_ref():
            refout = np.zeros(om * on, dtype=np.float32)
            ptrs = (C.c_void_p * len(ins))(*[x.ctypes.data for x in ins])
            assert ref["meqn"](iarr(*flat(nodes)), len(nodes), iarr(om, on, om, F32), ptrs, len(ins), refout.ctypes.data) == 0
            return refout
        # the node-by-node value in f32 (what the reference's portable path computes); the x86 JIT itself uses polynomial
        # tanh/exp approximations (seen: 1.3e-5 and 1e-3 off), so it only has to agree loosely
        A = [x.reshape(sh[1], sh[0]).T for x, sh in zip(ins, in_shapes)]
        exact = {"chain": lambda: np.tanh(A[0] + A[1]) * A[2], "bcast": lambda: np.maximum(A[0] * A[1] + A[2], 0),
                 "reduce": lambda: (A[0] * A[0]).sum(1, keepdims=True, dtype=np.float32), "ternary": lambda: A[0] - np.exp(A[1]) * A[2]}[name]()
        want = np.ascontiguousarray(exact.T.astype(np.float32)).ravel()
        refout, want_at = R.sampled(run_ref, want)
        assert np.allclose(refout, want_at, rtol=5e-3, atol=5e-3), name
        eq = build(nodes)
        fn = X.libxsmm_dispatch_meqn(eq, X.libxsmm_create_meqn_arg_shape(om, on, om, F32))
        assert fn, name
        for resident in (1, 0):
            if resident:
                d_in = [dev(x) for x in ins]; d_out = dev(np.zeros(om * on, dtype=np.float32))
                args = (X.MatrixArg * len(ins))(); out_ptr = d_out.data_ptr()
                for i, t in enumerate(d_in):
                    args[i].primary = t.data_ptr()
            else:
                hout = np.zeros(om * on, dtype=np.float32)
                args = (X.MatrixArg * len(ins))(); out_ptr = hout.ctypes.data
                for i, x in enumerate(ins):
                    args[i].primary = x.ctypes.data
            p = X.MeqnParam(); p.inputs = C.addressof(args); p.output.primary = out_ptr
            X.MEQN_FN(fn)(C.byref(p)); X.check()
            got = host(d_out, np.float32) if resident else hout
            assert np.allclose(got, want, rtol=2e-5, atol=2e-5), (name, m, n, resident, np.abs(got - want).max())


@pytest.mark.gpu
def test_gemm_nodes_are_declined():
    eq = build([("b", X.MELTW_TYPE_BINARY_MATMUL, F32, 0), ("arg", 0, 16, 16, 16, F32), ("arg", 1, 16, 16, 16, F32)])
    assert not X.libxsmm_dispatch_meqn(eq, X.libxsmm_create_meqn_arg_shape(16, 16, 16, F32))
