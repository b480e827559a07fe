"""GPU tests of the peer-memory exchange (csrc/p2p.cuh).  On one GPU the mailbox protocol runs with world = 1 (the kernels publish into and
gather from their own mailbox: same code path, no peer); with >= 2 GPUs the torchrun helper tools/check_multi_gpu.py compares the fused
exchange with NCCL and with the single-GPU result."""
import ctypes
import os
import subprocess
import sys
from ctypes import byref, c_void_p

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
Q = (1.0, 1.0, 5.0, 5.0, 0.2, 2.0)


def _mailbox(C, world=1, rank=0, cap=64):
    ctx, handle = c_void_p(), (ctypes.c_ubyte * 64)()
    C.call("b200sv_p2p_create", world, rank, cap, byref(ctx), handle)
    C.call("b200sv_p2p_connect", ctx, (ctypes.c_ubyte * (64 * world)).from_buffer_copy(bytes(handle) * world))
    return ctx


def test_publish_gather_roundtrip_and_epochs(cuda_lib):
    import torch
    from stochvolmodels_b200 import _capi as C
    ctx = _mailbox(C, cap=16)
    st = c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.zeros(16, dtype=torch.float64, device="cuda")
    for epoch in range(1, 8):                                   # crosses both slots several times
        vals = torch.arange(16, dtype=torch.float64, device="cuda") * epoch + 0.5
        C.call("b200sv_dev_p2p_publish", ctx, c_void_p(vals.data_ptr()), 16, st)
        if epoch % 3 == 0:                                      # a publish that is never gathered: the next publish must still be safe
            continue
        C.call("b200sv_dev_p2p_gather", ctx, 16, c_void_p(out.data_ptr()), st)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(out.cpu().numpy(), vals.cpu().numpy())
    with pytest.raises(C.B200svError):
        C.call("b200sv_dev_p2p_publish", ctx, c_void_p(out.data_ptr()), 17, st)      # exceeds the mailbox
    C.call("b200sv_p2p_destroy", ctx)
    with pytest.raises(C.B200svError):
        C.call("b200sv_p2p_create", 9, 0, 16, byref(c_void_p()), (ctypes.c_ubyte * 64)())   # world <= 8


@pytest.mark.parametrize("kinds,types", [(1, ["P", "P", "C", "C", "C"]), (0, ["IC", "P", "C", "IP", "C"])])
def test_fused_exchange_equals_plain_path_bitwise(cuda_lib, kinds, types):
    """slice -> payoff sums -> finalize with the exchange fused into the kernels == the same launches without a mailbox."""
    import torch
    from stochvolmodels_b200 import _capi as C, engine
    N, J = 200_000, 5
    pc = engine.logsv_params_c(*Q)
    strikes = torch.tensor([0.8, 0.9, 1.0, 1.1, 1.2], dtype=torch.float64, device="cuda")
    tcodes = torch.as_tensor(C.encode_types(np.array(types)), device="cuda")
    st = c_void_p(torch.cuda.current_stream().cuda_stream)
    ptr = lambda t: c_void_p(t.data_ptr())

    def chain(ctx):
        state = torch.empty((3, N), dtype=torch.float64, device="cuda")
        mom = torch.zeros(2, dtype=torch.float64, device="cuda")
        sums = torch.zeros(3 * J, dtype=torch.float64, device="cuda")
        out = torch.zeros((2, 2, J), dtype=torch.float64, device="cuda")
        for m in range(2):                                       # two maturities: epochs 1..4, both slots reused
            C.call("b200sv_dev_logsv_slice", ptr(state[0]), ptr(state[1]), ptr(state[2]), N, 0, int(m == 0), byref(pc), 1.0, 1, 40, 0.1 / 40, m,
                   1.0, 77, 0, ptr(mom), ctx, st)
            C.call("b200sv_dev_payoff_sums", ptr(state[0]), ptr(state[2]), N, 0, 0.1 * (m + 1), 1.0, ptr(strikes), ptr(tcodes), J, 1, kinds,
                   ptr(mom), ptr(sums), ctx, st)
            C.call("b200sv_dev_payoff_finalize", ptr(sums), J, 1.0, N, ptr(out[m, 0]), ptr(out[m, 1]), ctx, st)
        torch.cuda.synchronize()
        return out.cpu().numpy()

    plain = chain(None)
    ctx = _mailbox(C)
    fused = chain(ctx)
    C.call("b200sv_p2p_destroy", ctx)
    assert np.all(np.isfinite(fused)) and np.all(fused[:, 1] > 0)
    np.testing.assert_array_equal(fused, plain)
    small = _mailbox(C, cap=8)                                   # 3*J = 15 values do not fit
    with pytest.raises(C.B200svError, match="mailbox too small"):
        state = torch.zeros((3, 16), dtype=torch.float64, device="cuda")
        mom = torch.zeros(2, dtype=torch.float64, device="cuda")
        sums = torch.zeros(3 * J, dtype=torch.float64, device="cuda")
        C.call("b200sv_dev_payoff_sums", ptr(state[0]), ptr(state[2]), 16, 0, 0.1, 1.0, ptr(strikes), ptr(tcodes), J, 1, kinds, ptr(mom),
               ptr(sums), small, st)
    C.call("b200sv_p2p_destroy", small)


def test_gather_timeout_is_an_error_not_a_silent_nan(cuda_lib):
    """ADVICE r1: a peer that never publishes used to poison the prices with a quiet NaN.  Now the gather sets a status word that the host
    reads after the chain's copy back: b200sv_p2p_status reports the missing rank, CudaMcEngine.check_p2p raises P2pTimeout; the spin limit is
    configurable (2000 polls here: the test takes milliseconds, not the default 3 s)."""
    import torch
    from stochvolmodels_b200 import _capi as C, engine
    from stochvolmodels_b200.multi_gpu import CudaMcEngine, P2pTimeout
    ctx = _mailbox(C, cap=16)
    C.call("b200sv_p2p_set_spin_limit", ctx, 2000)
    st = c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.zeros(4, dtype=torch.float64, device="cuda")
    status = ctypes.c_uint(7)
    C.call("b200sv_p2p_status", ctx, byref(status), st)
    assert status.value == 0
    vals = torch.ones(4, dtype=torch.float64, device="cuda")
    C.call("b200sv_dev_p2p_publish", ctx, c_void_p(vals.data_ptr()), 4, st)          # a healthy exchange first
    C.call("b200sv_dev_p2p_gather", ctx, 4, c_void_p(out.data_ptr()), st)
    C.call("b200sv_p2p_status", ctx, byref(status), st)
    assert status.value == 0 and np.all(out.cpu().numpy() == 1.0)
    C.call("b200sv_debug_p2p_lose_publish", ctx)                                     # the "peer" (rank 0 of world 1) never arrives
    C.call("b200sv_dev_p2p_gather", ctx, 4, c_void_p(out.data_ptr()), st)
    C.call("b200sv_p2p_status", ctx, byref(status), st)
    assert status.value == 1 and np.all(np.isnan(out.cpu().numpy()))                 # bit 0 = rank 0 missing; values poisoned
    C.call("b200sv_p2p_status", ctx, byref(status), st)
    assert status.value == 0                                                         # reading clears it
    # the Python driver's check: an engine whose exchange timed out raises instead of returning NaN prices
    eng = CudaMcEngine("logsv", engine.logsv_params_c(*Q), 1000, 0, 0, 5)
    eng.p2p = ctx
    eng.check_p2p()                                                                   # clean: no raise
    C.call("b200sv_debug_p2p_lose_publish", ctx)
    sums = torch.zeros(15, dtype=torch.float64, device="cuda")
    eng.finalize(sums, 5, 1.0, 1000)                                                  # gathers the (never published) global sums
    with pytest.raises(P2pTimeout, match="rank"):
        eng.check_p2p()
    eng.p2p = None
    C.call("b200sv_p2p_destroy", ctx)


def test_two_gpu_exchange_vs_nccl_and_single_gpu(cuda_lib):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs: the peer-memory exchange is between two devices")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tools", "check_multi_gpu.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "p2p exchange == NCCL exchange bitwise: True" in r.stdout
