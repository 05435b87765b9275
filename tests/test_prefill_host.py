"""CPU-only checks of the prefill entry points (gfe_selscan_fwd_state, gfe_conv1d_silu_fwd_state): every bad argument is
rejected with a message before any launch.  Pointers are fake device addresses: nothing is dereferenced on the host."""
import ctypes

FAKE = 1 << 32           # 16-byte aligned fake device addresses, far apart
B, L, ED, N, K = 2, 64, 32, 16, 4


def _lib():
    from gfe_mamba_b200 import _native
    return _native, _native.lib()


def _args(nat):
    a = nat.SelscanArgs()
    a.batch, a.seqlen, a.d_inner, a.d_state = B, L, ED, N
    a.dtype = nat.GFE_F32
    for i, name in enumerate(("u", "delta", "Bm", "Cm", "A_log", "D", "out")):
        setattr(a, name, FAKE * (i + 1))
    a.u_rs = a.delta_rs = a.out_rs = ED
    a.B_rs = a.C_rs = N
    return a


def _fwd_state(lib, a, h0):
    return lib.gfe_selscan_fwd_state(ctypes.byref(a), ctypes.c_void_p(h0), None)


def test_selscan_fwd_state_rejects_bad_arguments():
    nat, lib = _lib()
    h0 = FAKE * 20
    a = nat.SelscanArgs()
    assert _fwd_state(lib, a, h0) == -1 and b"shape" in lib.gfe_last_error_string()
    a = _args(nat)
    a.seqlen = 0
    assert _fwd_state(lib, a, h0) == -1 and b"shape" in lib.gfe_last_error_string()
    a = _args(nat)
    a.u = None
    assert _fwd_state(lib, a, h0) == -1 and b"NULL" in lib.gfe_last_error_string()
    a = _args(nat)
    a.out = None
    assert _fwd_state(lib, a, h0) == -1 and b"out is NULL" in lib.gfe_last_error_string()
    a = _args(nat)
    a.ckpt, a.ckpt_bytes = FAKE * 30, 1 << 30
    assert _fwd_state(lib, a, h0) == -1 and b"ckpt" in lib.gfe_last_error_string()
    a = _args(nat)
    a.d_state = 8
    assert _fwd_state(lib, a, h0) == -3 and b"d_state" in lib.gfe_last_error_string()
    a = _args(nat)
    a.last_state = h0 + 4 * B * ED * N - 16          # the last 16 bytes of h0
    assert _fwd_state(lib, a, h0) == -1 and b"overlap" in lib.gfe_last_error_string()
    a.last_state = h0 - 16                           # ends inside h0
    assert _fwd_state(lib, a, h0) == -1 and b"overlap" in lib.gfe_last_error_string()
    a = _args(nat)
    assert _fwd_state(lib, a, h0 + 8) == -1 and b"aligned" in lib.gfe_last_error_string()


def test_conv1d_fwd_state_rejects_bad_arguments():
    nat, lib = _lib()
    x, w, u, cin, cout = (FAKE * i for i in range(1, 6))

    def call(x=x, w=w, u=u, cin=cin, cout=cout, L=L, K=K):
        return lib.gfe_conv1d_silu_fwd_state(x, ED, ED, w, None, cin, cout, u, ED, ED, B, L, ED, K, nat.GFE_F32, None)

    assert call(x=None) == -1 and b"NULL" in lib.gfe_last_error_string()
    assert call(u=None) == -1 and b"NULL" in lib.gfe_last_error_string()
    assert call(L=0) == -1 and b"shape" in lib.gfe_last_error_string()
    win = 4 * B * ED * (K - 1)
    assert call(cout=cin + win - 4) == -1 and b"overlap" in lib.gfe_last_error_string()
    assert call(cin=cout + win - 4) == -1 and b"overlap" in lib.gfe_last_error_string()
    assert call(K=5, cout=None) == -3 and b"d_conv" in lib.gfe_last_error_string()
    assert call(K=1, cin=None, cout=None) == -3 and b"d_conv" in lib.gfe_last_error_string()
