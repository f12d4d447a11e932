"""Callable losses on 6-8 qubits, host side: the argument checks of cpf_adjoint_from_cotangent on 6-8 qubit programs
(made before any device work, so fake pointers are never dereferenced), the chunk arithmetic of the host-driven loop,
and the refusal text of the fused HS and relative-phase losses, which stay limited to n <= 5."""
import ctypes as C

import pytest
import torch

from cpflow_b200 import _lib as L
from cpflow_b200.ansatz import Ansatz
from cpflow_b200.optimization import TORCH_LOSS_U_BYTES, chunk_ranges, torch_loss_chunk
from cpflow_b200.topology import chain_layer, fill_layers


def _chain(n, K=6):
    return Ansatz(n, "cp", fill_layers(chain_layer(n), K)).program


def _err():
    return L.load().cpf_last_error().decode()


@pytest.mark.parametrize("n", [6, 7, 8])
def test_cotangent_argument_checks(lib, n):
    prog = _chain(n)
    f = lib.cpf_adjoint_from_cotangent
    fake = C.c_void_p(256)
    assert f(None, L.F32, 4, fake, fake, fake, None) == -1
    assert f(prog._h, L.F32, -1, fake, fake, fake, None) == -1
    for args in ((None, fake, fake), (fake, None, fake), (fake, fake, None)):
        assert f(prog._h, L.F64, 4, *args, None) == -1 and "NULL argument" in _err()
    assert f(prog._h, 7, 4, fake, fake, fake, None) == -1 and "unknown dtype" in _err()
    # batch 0 is a no-op, whatever the pointers
    assert f(prog._h, L.F32, 0, None, None, None, None) == 0


@pytest.mark.parametrize("n", [6, 7, 8])
@pytest.mark.parametrize("kind", [L.LOSS_HS, L.LOSS_RELPHASE])
def test_fused_full_unitary_refusal_text(lib, n, kind):
    prog = _chain(n)
    spec = L.CpfLossSpec(kind, 1, 0)
    assert lib.cpf_loss_grad(prog._h, C.byref(spec), None, L.F32, 4, C.c_void_p(16), C.c_void_p(8), None, None,
                             None) == -2
    assert "full-unitary losses need n <= 5" in _err()
    b = C.c_int64()
    assert lib.cpf_workspace_bytes(prog._h, kind, L.F32, 4, C.byref(b)) == -2
    assert "full-unitary losses need n <= 5" in _err()


def test_chunk_ranges():
    assert chunk_ranges(10, None) == [(0, 10)]
    assert chunk_ranges(10, 10) == [(0, 10)]
    assert chunk_ranges(10, 64) == [(0, 10)]
    assert chunk_ranges(10, 4) == [(0, 4), (4, 8), (8, 10)]
    assert chunk_ranges(37, 32) == [(0, 32), (32, 37)]
    assert chunk_ranges(3, 1) == [(0, 1), (1, 2), (2, 3)]
    for B, c in ((1000, 7), (4096, 4096), (4097, 4096)):
        r = chunk_ranges(B, c)
        assert r[0][0] == 0 and r[-1][1] == B and all(a[1] == b[0] for a, b in zip(r, r[1:]))
        assert all(0 < j - i <= c for i, j in r)
    with pytest.raises(ValueError):
        chunk_ranges(10, 0)


def test_torch_loss_chunk():
    for n in (2, 3, 4, 5):
        assert torch_loss_chunk(_chain(n, 2), torch.float32) is None
        assert torch_loss_chunk(_chain(n, 2), torch.float64) is None
    for n in (6, 7, 8):
        N = 1 << n
        for dt, cbytes in ((torch.float32, 8), (torch.float64, 16)):
            c = torch_loss_chunk(_chain(n, 2), dt)
            assert c * N * N * cbytes <= TORCH_LOSS_U_BYTES < (c + 1) * N * N * cbytes
    assert torch_loss_chunk(_chain(8, 2), torch.float32) == 4096
    assert torch_loss_chunk(_chain(8, 2), torch.float64) == 2048
