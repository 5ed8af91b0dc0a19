"""Host-side argument checks of qsae_bsae_backward and its workspace query (no device needed: every call below fails
or answers before anything touches the GPU), and the model switch that selects it."""
import ctypes as C

from quantizedsae_b200 import _lib


def _ws(lib, B, H, D, k, n_bits):
    n = C.c_size_t(0)
    rc = lib.qsae_bsae_backward_workspace_bytes(B, H, D, k, n_bits, C.byref(n))
    return rc, n.value


def test_workspace_query_checks_shapes():
    lib = _lib.load()
    assert _ws(lib, 16, 2048, 64, 32, 4)[0] == 0 and _ws(lib, 16, 2048, 64, 32, 4)[1] > 0
    assert _ws(lib, 0, 2048, 64, 32, 4)[0] == 0                                        # empty batch
    assert lib.qsae_bsae_backward_workspace_bytes(16, 2048, 64, 32, 4, None) == -1
    assert b"null pointer" in lib.qsae_last_error()
    bad = {
        (-1, 2048, 64, 32, 4): (-1, b"negative batch"),
        (16, 2048, 520, 32, 4): (-1, b"multiple of 8"),                                 # D > 512
        (16, 2048, 60, 32, 4): (-1, b"multiple of 8"),                                  # D % 8
        (16, 2048, 0, 32, 4): (-1, b"multiple of 8"),
        (16, 0, 64, 32, 4): (-1, b"positive"),                                          # H = 0
        (16, 2048, 64, 32, 0): (-1, b"n_bits"),
        (16, 2048, 64, 32, 9): (-1, b"n_bits"),
        (16, 2048, 64, 0, 4): (-1, b"k must be >= 1"),
        (16, 2048, 64, 4096, 4): (-5, b"out of range"),                                 # k > H
        (16, 8192, 64, 4097, 4): (-1, b"QSAE_MAX_K_LARGE"),
        (1 << 20, 4096, 64, 4096, 4): (-1, b"2^31"),                                    # B k >= 2^31
    }
    for args, (rc, text) in bad.items():
        assert _ws(lib, *args)[0] == rc, args
        assert text in lib.qsae_last_error(), (args, lib.qsae_last_error())


def test_workspace_is_monotone_in_batch_and_k():
    lib = _lib.load()
    for H, D, nb in ((1000, 8, 1), (32768, 512, 4), (1 << 20, 64, 8)):
        prev = 0
        for B in (1, 37, 4096, 65536):
            rc, n = _ws(lib, B, H, D, 32, nb)
            assert rc == 0 and n >= prev, (H, B)
            prev = n
        prev = 0
        for k in (1, 32, 65, 500, 1000):
            rc, n = _ws(lib, 4096, H, D, k, nb)
            assert rc == 0 and n >= prev, (H, k)
            prev = n
    # the b_sae backward uses the baseline_sae backward's regions: n_bits does not change the size
    assert _ws(lib, 4096, 32768, 512, 32, 1)[1] == _ws(lib, 4096, 32768, 512, 32, 8)[1]
    n = C.c_size_t(0)
    assert lib.qsae_baseline_backward_workspace_bytes(4096, 32768, 512, 32, C.byref(n)) == 0
    assert _ws(lib, 4096, 32768, 512, 32, 4)[1] == n.value


def test_backward_checks_arguments():
    lib = _lib.load()
    B, H, D, k, nb = 16, 2048, 64, 32, 4
    need = _ws(lib, B, H, D, k, nb)[1]
    p = 1 << 20           # never dereferenced: every call below fails its host-side checks

    def args(**kw):
        a = dict(x=p, vals=p, idx=p, g=p, rows=p, logits=p, q=0.5, gp_dev=None, gp_host=0.1, w_enc=p, B=B, H=H, D=D, k=k,
                 n_bits=nb, gwe=p, gbe=p, glog=p, gbd=p, gx=None, ws=p, ws_bytes=need, stream=None)
        a.update(kw)
        return list(a.values())

    def call(**kw):
        return lib.qsae_bsae_backward(*args(**kw))

    assert call(ws_bytes=need - 1) == -2                                                 # workspace too small
    assert b"workspace" in lib.qsae_last_error()
    for name in ("gwe", "gbe", "glog", "gbd"):
        assert call(**{name: None}) == -1, name
        assert b"null gradient" in lib.qsae_last_error()
    for name in ("x", "vals", "idx", "g", "rows", "ws"):
        assert call(**{name: None}) == -1, name
        assert b"null pointer" in lib.qsae_last_error()
    assert call(logits=None) == -1 and b"null pointer" in lib.qsae_last_error()
    assert call(logits=None, B=0) == -1                                                  # the polarize term needs the logits
    for name in ("x", "g", "rows", "logits", "w_enc", "gwe", "glog", "ws"):
        assert call(**{name: p + 4}) == -1, name
        assert b"16-byte" in lib.qsae_last_error()
    assert call(gx=p + 4) == -1 and b"16-byte" in lib.qsae_last_error()
    assert call(w_enc=None, gx=p) == -1 and b"W_enc" in lib.qsae_last_error()
    assert call(D=520) == -1 and b"multiple of 8" in lib.qsae_last_error()
    assert call(n_bits=0) == -1 and b"n_bits" in lib.qsae_last_error()
    assert call(n_bits=9) == -1 and b"n_bits" in lib.qsae_last_error()
    assert call(k=0) == -1
    assert call(k=H + 1) == -5
    assert call(B=-1) == -1 and b"negative batch" in lib.qsae_last_error()


def test_switch_defaults_off_and_is_not_state():
    import quantizedsae_b200 as Q

    m = Q.BinarySAE(16, 64, 4.0, 4)
    assert m.deterministic is False
    assert all("deterministic" not in key for key in m.state_dict())
