"""Host side of the ordered (bitwise-reproducible) entry points: invalid arguments and short workspaces come back as -1 before
any launch, and the split-K workspace query answers without a device."""
import ctypes as C

from multimodalsum_b200 import _lib, ops

P = C.c_void_p(4096)
i32, i64, f32, u32, u64 = C.c_int32, C.c_int64, C.c_float, C.c_uint32, C.c_uint64


def _call_all_bad(fn, ok, bads):
    order = list(ok)
    for bad in bads:
        args = dict(ok, **bad)
        assert fn(*[args[k] for k in order]) == -1, bad


def test_gemm_ordered_workspace_query():
    L = _lib.lib()
    n = i64(-5)
    assert L.mmsum_gemm_ordered_workspace(None, C.byref(n)) == -1
    assert L.mmsum_gemm_ordered_workspace(C.byref(_lib.GemmArgs(M=128, N=128, K=64)), None) == -1
    # 1024 x 1024 x 18432 wgrad on 148 SMs: 4 n-tiles x 8 m-tiles, split 4 ways -> 4 regions of 1024 x 1024 fp32
    assert ops.gemm_workspace_elems(1024, 1024, 18432) == 4 * 1024 * 1024
    assert ops.gemm_workspace_elems(4096, 1024, 18432) == 0            # 128 tiles: one split, nothing to order
    assert ops.gemm_workspace_elems(1000, 1000, 64) == 0               # one k-block
    # M rounds up to whole 128-row tiles, N to a 16-byte row pitch
    need = ops.gemm_workspace_elems(1000, 1002, 18432)
    assert need > 0 and need % (1024 * 1004) == 0
    # non-accumulating or bf16 calls have one writer per element
    a = _lib.GemmArgs(M=1024, N=1024, K=18432, a_mn_major=1, b_mn_major=1)
    assert L.mmsum_gemm_ordered_workspace(C.byref(a), C.byref(n)) == 0 and n.value == 0


def test_gemm_ordered_rejects_invalid_arguments_on_the_host():
    L = _lib.lib()
    ok = dict(A=4096, B=4096, D=4096, lda=1024, ldb=1024, ldd=1024, M=1024, N=1024, K=18432, a_mn_major=1, b_mn_major=1,
              out_f32=1, accumulate=1)
    need = ops.gemm_workspace_elems(1024, 1024, 18432)
    a = _lib.GemmArgs(**ok)
    assert L.mmsum_gemm_bf16_ordered(None, P, i64(need), None) == -1
    assert L.mmsum_gemm_bf16_ordered(C.byref(a), None, i64(need), None) == -1                    # no workspace
    assert L.mmsum_gemm_bf16_ordered(C.byref(a), P, i64(need - 1), None) == -1                   # too small
    assert L.mmsum_gemm_bf16_ordered(C.byref(a), C.c_void_p(4100), i64(need), None) == -1       # not 16-byte aligned
    for bad in (dict(M=0), dict(A=0), dict(accumulate=0, splits=4), dict(act=2)):
        assert L.mmsum_gemm_bf16_ordered(C.byref(_lib.GemmArgs(**dict(ok, **bad))), P, i64(need), None) == -1, bad


def test_add_ln_bwd_ordered_rejects_invalid_arguments_on_the_host():
    L = _lib.lib()
    ok = dict(d1=P, d2=None, res=P, y=P, gamma=P, mean=P, rstd=P, dres=P, dy=C.c_void_p(8192), dgamma=P, dbeta=P, rows=18432,
              d_model=1024, p_drop=f32(0.1), seed=u64(1), sid=u32(2), step_dev=None, ws=P, ws_elems=i64(ops.ADD_LN_BWD_WORKSPACE),
              stream=None)
    bads = [dict(d1=None), dict(res=None), dict(y=None), dict(dres=None), dict(dy=None), dict(dgamma=None), dict(dbeta=None),
            dict(rows=0), dict(d_model=768), dict(dy=P), dict(ws=None), dict(ws_elems=i64(444 * 2048 - 1))]
    _call_all_bad(L.mmsum_add_ln_bwd_ordered, ok, bads)


def test_colsum_ordered_rejects_invalid_arguments_on_the_host():
    L = _lib.lib()
    ok = dict(x=P, ld=i64(3072), rows=18432, N=3072, out=P, ws=P, ws_elems=i64(ops.colsum_workspace(3072)), stream=None)
    bads = [dict(x=None), dict(out=None), dict(ws=None), dict(rows=0), dict(N=0), dict(N=3071), dict(ld=i64(3076)),
            dict(ws_elems=i64(49 * 3072 - 1))]                                # 12 column blocks x 49 row chunks
    _call_all_bad(L.mmsum_colsum_ordered, ok, bads)


def test_embed_ln_bwd_ordered_rejects_invalid_arguments_on_the_host():
    L = _lib.lib()
    rows, S, V = 18432, 128, 50265
    ok = dict(dout=P, dout2=None, ids=P, E=P, Pos=P, rd=P, remb=P, gamma=P, mean=P, rstd=P, dE=P, dP=P, dremb=P, dgamma=P,
              dbeta=P, dz=P, rows=rows, S=S, d_model=1024, pad=1, p_drop=f32(0.1), seed=u64(1), sid=u32(3), step_dev=None, V=V,
              ws=P, ws_elems=i64(ops.embed_ln_bwd_workspace(rows, S, V)), stream=None)
    exact = 576 * 2048 + S * 1024 + 2048 * 288 + V + 1 + 2 * rows  # 576 CTAs of 32 rows (the header's bound assumes 592), 288 tiles
    bads = [dict(dout=None), dict(ids=None), dict(E=None), dict(dE=None), dict(dP=None), dict(dz=None), dict(dgamma=None),
            dict(remb=None), dict(dremb=None), dict(rows=0), dict(S=0), dict(rows=rows - 1), dict(d_model=512), dict(V=0),
            dict(V=1 << 22), dict(ws=None), dict(ws_elems=i64(exact - 1))]
    _call_all_bad(L.mmsum_embed_ln_bwd_ordered, ok, bads)
    # the encoder (no rating embedding) needs neither remb nor dremb
    enc = dict(ok, rd=None, remb=None, dremb=None)
    _call_all_bad(L.mmsum_embed_ln_bwd_ordered, enc, [dict(ws_elems=i64(exact - 1)), dict(ids=None)])
