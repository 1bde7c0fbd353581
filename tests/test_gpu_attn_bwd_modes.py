"""Every kernel variant of the tcgen05 attention backward (progen_local_attn_bwd_tc_ex `mode`) on the same seeded inputs:
against the mode-2 kernels (mode 3 only changes how the gradient tiles are stored: same values up to bf16 rounding of
the same fp32 numbers) and against the fp32 CUDA-core backward followed by the separate rotary backward kernel.
Shapes: one sequence batch of the cfg2 and cfg3 attention shapes, and seq_len == window (window-0 items only)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

MODES = (0, 1, 2, 3)
# per-part bounds of the existing bf16 attention-backward tests (test_gpu_attn_mma.py::test_local_attn_tcgen05_bwd)
REL_FRO, REL_MAX = 2e-2, 5e-2


def _run_tc(L, qkv, out, dout, lse, B, n, w, h, mode, tables):
    sin, cos, sin_t, cos_t = tables
    dqkv = torch.full_like(qkv, float('nan'))
    delta = torch.full((qkv.shape[0], h), float('nan'), device=qkv.device)
    ptr = lambda t: t.data_ptr() if t is not None else 0
    L.check(L.load().progen_local_attn_bwd_tc_ex(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(),
                                                 dqkv.data_ptr(), delta.data_ptr(), ptr(sin), ptr(cos), ptr(sin_t), ptr(cos_t),
                                                 B, n, w, h, 64, mode, L.stream()))
    torch.cuda.synchronize()
    assert torch.isfinite(delta).all()
    return dqkv


@pytest.mark.parametrize('cfg', [(2, 1024, 256, 8), (1, 2048, 512, 16), (2, 256, 256, 4)], ids=['cfg2', 'cfg3', 'n_eq_w'])
@pytest.mark.parametrize('rotary', [False, True])
def test_attn_bwd_modes_agree(cfg, rotary):
    from progen_b200 import lib as L
    from gemm_cases import rotary_tables
    L.require_device()
    B, n, w, h = cfg
    dh, dev = 64, 'cuda'
    T, I = B * n, h * dh
    g = torch.Generator(device=dev).manual_seed(11 * n + w + h)
    qkv = (torch.randn(T, 3 * I, generator=g, device=dev) * 1.5).bfloat16()
    dout = torch.randn(T, I, generator=g, device=dev).bfloat16()
    out = torch.empty(T, I, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(T, h, device=dev)
    L.check(L.load().progen_local_attn_fwd_tc(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), B, n, w, h, dh, L.stream()))
    sin, cos = rotary_tables(n, dh, dev)
    tables = (sin, cos, sin.t().contiguous(), cos.t().contiguous()) if rotary else (None, None, None, None)

    # fp32 reference: CUDA-core forward + backward on the same (exactly up-cast) inputs, then the rotary backward pass
    q32, do32 = qkv.float(), dout.float()
    o32, lse32, d32 = torch.empty(T, I, device=dev), torch.empty(T, h, device=dev), torch.empty(T, h, device=dev)
    ref = torch.empty_like(q32)
    L.check(L.load().progen_local_attn_fwd_simt(q32.data_ptr(), o32.data_ptr(), lse32.data_ptr(), L.F32, B, n, w, h, dh, L.stream()))
    L.check(L.load().progen_local_attn_bwd_simt(q32.data_ptr(), o32.data_ptr(), do32.data_ptr(), lse32.data_ptr(), ref.data_ptr(),
                                                d32.data_ptr(), L.F32, B, n, w, h, dh, L.stream()))
    if rotary:
        L.check(L.load().progen_rotary_bwd(ref.data_ptr(), 3 * I, L.F32, sin.data_ptr(), cos.data_ptr(), T, 3 * I, n, dh, L.stream()))
    torch.cuda.synchronize()
    ref = ref.double()

    res = {m: _run_tc(L, qkv, out, dout, lse, B, n, w, h, m, tables) for m in MODES}
    if rotary:       # mode 3 given only the [n, 32] tables (what progen_local_attn_bwd_tc passes)
        res['3rm'] = _run_tc(L, qkv, out, dout, lse, B, n, w, h, 3, (sin, cos, None, None))

    for m, d in res.items():
        assert torch.isfinite(d.float()).all(), m
        for part, name in enumerate(('dq', 'dk', 'dv')):
            a_ = d.double()[:, part * I:(part + 1) * I]
            r_ = ref[:, part * I:(part + 1) * I]
            rel = (a_ - r_).norm().item() / r_.norm().item()
            assert rel < REL_FRO, (m, name, rel)
            assert (a_ - r_).abs().max().item() < REL_MAX * max(1.0, r_.abs().max().item()), (m, name)

    # mode 3 vs mode 2: the same fp32 accumulators, rounded to bf16 once; at most one bf16 step apart where the
    # un-rotation's multiply-adds are contracted differently
    base = res[2].double()
    for m in (3, '3rm') if rotary else (3,):
        diff = (res[m].double() - base).abs()
        assert (diff <= base.abs() * 2.0 ** -7 + 1e-30).all(), (m, diff.max().item())
    if not rotary:
        assert torch.equal(res[3], res[2])
