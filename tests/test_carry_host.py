"""CPU-only checks of the entry points for training from a carried state (gfe_selscan_fwd_carry, gfe_selscan_bwd_carry,
gfe_conv1d_silu_bwd_carry): every bad argument is rejected with a message before any launch.  Pointers are fake device
addresses: nothing is dereferenced on the host."""
import ctypes

FAKE = 1 << 32           # 16-byte aligned fake device addresses, far apart
B, L, ED, N, K = 2, 64, 32, 16, 4
STATE = 4 * B * ED * N   # bytes of a (B, ED, N) fp32 state


def _lib():
    from gfe_mamba_b200 import _native
    return _native, _native.lib()


def _args(nat, bwd=False):
    a = nat.SelscanArgs()
    a.batch, a.seqlen, a.d_inner, a.d_state = B, L, ED, N
    a.dtype = nat.GFE_F32
    names = ("u", "delta", "Bm", "Cm", "A_log", "D", "out")
    if bwd:
        names += ("dout", "du", "ddelta", "dBm", "dCm", "dA_log", "dD")
        a.ckpt, a.ckpt_bytes = FAKE * 40, 1 << 30
    for i, name in enumerate(names):
        setattr(a, name, FAKE * (i + 1))
    a.u_rs = a.delta_rs = a.out_rs = a.dout_rs = a.du_rs = a.ddelta_rs = ED
    a.u_bs = a.delta_bs = a.out_bs = a.dout_bs = a.du_bs = a.ddelta_bs = L * ED
    a.B_rs = a.C_rs = a.dB_rs = a.dC_rs = N
    a.B_bs = a.C_bs = a.dB_bs = a.dC_bs = L * N
    return a


def _err(lib):
    return lib.gfe_last_error_string()


def test_selscan_fwd_carry_rejects_bad_arguments():
    nat, lib = _lib()
    h0 = FAKE * 20
    call = lambda a, h: lib.gfe_selscan_fwd_carry(ctypes.byref(a), ctypes.c_void_p(h), None)
    a = _args(nat)
    a.out = None
    assert call(a, h0) == -1 and b"out is NULL" in _err(lib)
    a = _args(nat)
    a.ckpt, a.ckpt_bytes = FAKE * 30, 16                  # a checkpoint is allowed here, but it must be large enough
    assert call(a, h0) == -4 and b"checkpoint buffer too small" in _err(lib)
    a = _args(nat)
    assert call(a, h0 + 8) == -1 and b"aligned" in _err(lib)
    a.last_state = h0 + STATE - 16
    assert call(a, h0) == -1 and b"overlap" in _err(lib)
    a = _args(nat)
    a.d_state = 8
    assert call(a, h0) == -3 and b"d_state" in _err(lib)


def test_selscan_fwd_state_still_refuses_checkpoints():
    nat, lib = _lib()
    a = _args(nat)
    a.ckpt, a.ckpt_bytes = FAKE * 30, 1 << 30
    assert lib.gfe_selscan_fwd_state(ctypes.byref(a), None, None) == -1 and b"ckpt" in _err(lib)


def test_selscan_bwd_carry_rejects_bad_arguments():
    nat, lib = _lib()
    dlast, dh0 = FAKE * 50, FAKE * 60
    call = lambda a, dl=dlast, dh=dh0: lib.gfe_selscan_bwd_carry(ctypes.byref(a), ctypes.c_void_p(dl), ctypes.c_void_p(dh), None)
    a = _args(nat, bwd=True)
    a.ckpt, a.ckpt_bytes = None, 0
    assert call(a) == -4 and b"checkpoints" in _err(lib)
    a = _args(nat, bwd=True)
    a.du = None
    assert call(a) == -1 and b"NULL gradient" in _err(lib)
    a = _args(nat, bwd=True)
    assert call(a, dl=dlast + 8) == -1 and b"aligned" in _err(lib)
    assert call(a, dh=dh0 + 4) == -1 and b"aligned" in _err(lib)
    assert call(a, dl=0, dh=dh0 + 8) == -1 and b"aligned" in _err(lib)
    # dh0 against dlast and every output; NULL dlast or NULL dh0 are not checked against anything
    assert call(a, dl=dh0 + STATE - 16) == -1 and b"overlap" in _err(lib)
    assert call(a, dl=dh0 - STATE + 16) == -1 and b"overlap" in _err(lib)
    for name, size in (("du", 4 * B * L * ED), ("ddelta", 4 * B * L * ED), ("dBm", 4 * B * L * N), ("dCm", 4 * B * L * N),
                       ("dA_log", 4 * ED * N), ("dD", 4 * ED)):
        a = _args(nat, bwd=True)
        setattr(a, name, dh0 + STATE - 16)               # starts inside dh0
        assert call(a) == -1 and b"overlap" in _err(lib), name
        setattr(a, name, dh0 - size + 16)                # ends inside dh0
        assert call(a) == -1 and b"overlap" in _err(lib), name
    a = _args(nat, bwd=True)
    a.ddt_bias = dh0
    assert call(a) == -1 and b"overlap" in _err(lib)
    a = _args(nat, bwd=True)
    a.z, a.z_rs, a.z_bs = FAKE * 70, ED, L * ED
    a.dz, a.dz_rs, a.dz_bs = dh0 - 4 * B * L * ED + 16, ED, L * ED
    assert call(a) == -1 and b"overlap" in _err(lib)


def test_conv1d_bwd_carry_rejects_bad_arguments():
    nat, lib = _lib()
    x, w, du, dx, dw, cin, dcin, ws = (FAKE * i for i in range(1, 9))

    def call(x=x, du=du, dx=dx, dw=dw, cin=cin, dcin=dcin, L=L, K=K, ws=ws, nws=1 << 30):
        return lib.gfe_conv1d_silu_bwd_carry(x, ED, ED, w, None, cin, du, ED, ED, dx, ED, ED, dw, None, dcin,
                                             B, L, ED, K, nat.GFE_F32, ws, nws, None)

    assert call(x=None) == -1 and b"NULL" in _err(lib)
    assert call(dx=None) == -1 and b"NULL" in _err(lib)
    assert call(L=0) == -1 and b"shape" in _err(lib)
    assert call(ws=None) == -4 and b"workspace" in _err(lib)
    win = 4 * B * ED * (K - 1)
    assert call(dcin=cin + win - 4) == -1 and b"overlap" in _err(lib)
    assert call(cin=dcin + win - 4) == -1 and b"overlap" in _err(lib)
    assert call(K=5, dcin=None) == -3 and b"d_conv" in _err(lib)
