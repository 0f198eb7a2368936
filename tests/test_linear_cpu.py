"""Argument checks of sfod_linear_3xtf32 (host only): every refusal happens before any launch."""
from sfod_b200 import _lib


def test_linear_3xtf32_refuses_before_any_launch():
    L = _lib.lib()
    launches = L.sfod_debug_launch_count()
    M, N, K = 16000, 1024, 25088
    need = L.sfod_linear_3xtf32_workspace_bytes(M, N, K)
    assert need >= 2 * 4 * (M * K + N * K)                           # hi and lo planes of x and W
    assert L.sfod_linear_3xtf32_workspace_bytes(-1, N, K) == 0
    x, w, b, y, ws = 0x10000, 0x20000, 0x30000, 0x40000, 0x50000      # never dereferenced: every call below is refused
    args = dict(x=x, M=M, K=K, w=w, N=N, bias=b, act=1, y=y, ws=ws, nbytes=need)

    def call(**over):
        a = {**args, **over}
        return L.sfod_linear_3xtf32(a["x"], a["M"], a["K"], a["w"], a["N"], a["bias"], a["act"], a["y"], a["ws"], a["nbytes"], None)

    assert call(x=None) == 1 and call(w=None) == 1 and call(y=None) == 1
    assert call(M=-1) == 1 and call(K=0) == 1 and call(N=0) == 1 and call(act=2) == 1
    assert call(K=25090) == 3 and call(N=1000) == 3 and call(M=65536 * 128) == 3     # SFOD_ERR_UNSUPPORTED
    assert call(x=x + 4) == 4 and call(w=w + 8) == 4 and call(y=y + 4) == 4 and call(ws=ws + 4) == 4   # SFOD_ERR_ALIGNMENT
    assert call(nbytes=need - 1) == 2 and call(ws=None) == 2                           # SFOD_ERR_WORKSPACE_TOO_SMALL
    assert call(M=0) == 0                                                              # empty: nothing to launch
    assert L.sfod_debug_launch_count() == launches
