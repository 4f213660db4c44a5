"""Argument checks of the batched MPPI entry points (include/odg_mppi.h) that need no device: each refusal returns
ODG_ERR_INVALID with a message before any CUDA call. The refusals that need live handles are in test_gpu_mppi_batched.py."""
import ctypes as C

INVALID = -1


def test_batched_mppi_refuses_bad_arguments_without_a_device():
    from opendog_b200 import lib
    L = lib.load()
    P = C.c_void_p(0x10000)                 # never dereferenced: every call below is refused before it touches memory
    assert L.odg_mppi_broadcast(None, None, 0, 1, None) == INVALID and b"odg_mppi_broadcast" in L.odg_last_error()
    assert L.odg_mppi_broadcast(P, None, 0, 1, None) == INVALID and b"null handle" in L.odg_last_error()
    assert L.odg_mppi_broadcast(None, P, 0, 1, None) == INVALID and b"null handle" in L.odg_last_error()
    assert L.odg_mppi_rollout_groups(None, 2, P, 0.3, 4, 0, 0, None, 100.0, P, P, None) == INVALID
    assert b"odg_mppi_rollout_groups" in L.odg_last_error()

    def reduce(T=3, G=2, S=16, A=8, lam=1.0, cost=P, act=P, out=P):
        rc = L.odg_mppi_reduce_groups(cost, act, T, G, S, A, lam, out, None, None)
        return rc, L.odg_last_error()
    for kw in (dict(G=0), dict(G=-1), dict(S=0), dict(S=12001), dict(T=0), dict(A=0), dict(lam=0.0), dict(lam=float("nan")),
               dict(cost=None), dict(act=None), dict(out=None)):
        rc, msg = reduce(**kw)
        assert rc == INVALID and b"odg_mppi_reduce_groups" in msg and b"12000" in msg, kw
