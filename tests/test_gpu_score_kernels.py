"""GPU parity of the three tcgen05 scoring GEMMs (tcar_score_fwd / _bwd_q / _bwd_i) called through the C ABI.

The checker here is a plain torch fp32/fp64 matmul over the SAME bf16-rounded operands (this is a floating-point
kernel, so a torch reference is the right unit-level oracle; end-to-end parity against oracle/ lives in
test_gpu_parity.py).  Tolerances: fp32 accumulation of bf16 products -> rtol 2e-3 on sums, bf16 output rounding
(2^-8) on E.
"""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

KEXT, QROWS = 640, 512


def e_to_blocked(E):
    """logical [512, n_pad] -> stored [n_pad/8][512][8] (include/tcar_b200.h, tcar_score_fwd)."""
    return E.view(QROWS, -1, 8).permute(1, 0, 2).contiguous()


def e_from_blocked(Eb, n_pad):
    return Eb.view(n_pad // 8, QROWS, 8).permute(1, 0, 2).reshape(QROWS, n_pad)


def _mk(B, N, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n_pad = (N + 255) // 256 * 256
    Q = torch.zeros(QROWS, KEXT, device="cuda", dtype=torch.bfloat16)
    Q[:B] = (torch.randn(B, KEXT, device="cuda", generator=g) * 0.5).bfloat16()
    I = torch.zeros(n_pad, KEXT, device="cuda", dtype=torch.bfloat16)
    I[:N] = (torch.randn(N, KEXT, device="cuda", generator=g) * 0.1).bfloat16()
    c = torch.randn(QROWS, device="cuda", generator=g) * 0.3
    return Q, I, c, n_pad


def _fwd(native, Q, I, c, B, N, n_pad, mode, cluster):
    tiles = native.lib().tcar_score_fwd_tiles(n_pad)
    part = torch.zeros(tiles, QROWS, device="cuda")
    E = torch.full((QROWS, n_pad), float("nan"), device="cuda", dtype=torch.bfloat16) if mode == 0 else None
    cm = torch.full((QROWS, n_pad // 8), float("nan"), device="cuda") if mode == 1 else None
    tmx = torch.full((QROWS, n_pad // 128), float("nan"), device="cuda") if mode == 1 else None
    native.call("tcar_score_fwd", native.ptr(Q), native.ptr(I), native.ptr(c), native.ptr(E), native.ptr(part),
                native.ptr(cm), native.ptr(tmx), B, N, n_pad, mode, cluster)
    torch.cuda.synchronize()
    if mode == 1:
        # the per-128-item maxima are the maxima of their 16 chunk maxima
        assert torch.equal(tmx[:B], cm[:B].view(B, -1, 16).max(-1).values)
    return (e_from_blocked(E, n_pad) if E is not None else None), part, cm


@pytest.mark.parametrize("cluster", [1, 2, 4, -2])
@pytest.mark.parametrize("B,N", [(512, 5000), (300, 2333), (64, 20000), (1, 300), (129, 70000)])
def test_score_fwd_train(native, cluster, B, N):
    Q, I, c, n_pad = _mk(B, N, 7 + B + N)
    E, part, _ = _fwd(native, Q, I, c, B, N, n_pad, 0, cluster)
    S = Q[:B].float() @ I[:N].float().t()
    ref = torch.exp(S - c[:B, None])
    got = E[:B, :N].float()
    err = ((got - ref).abs() / (ref.abs() + 1e-6)).max().item()
    assert err < 1.2e-2, f"E rel err {err}"
    assert (E[:B, N:].float() == 0).all(), "padded item columns must be exactly zero"
    kpad = (B + 63) // 64 * 64
    assert (E[B:kpad].float() == 0).all(), "K-padding rows must be exactly zero"
    rs = part.sum(0)[:B]
    rerr = ((rs - ref.sum(1)).abs() / ref.sum(1)).max().item()
    assert rerr < 2e-3, f"rowsum rel err {rerr}"


@pytest.mark.parametrize("cluster", [1, 4, -2])
def test_score_fwd_eval_chunkmax(native, cluster):
    B, N = 257, 7001
    Q, I, c, n_pad = _mk(B, N, 99)
    _, part, cm = _fwd(native, Q, I, c, B, N, n_pad, 1, cluster)
    S = Q[:B].float() @ I[:N].float().t()
    Sp = torch.full((B, (N + 7) // 8 * 8), float("-inf"), device="cuda")
    Sp[:, :N] = S
    ref = Sp.view(B, -1, 8).max(-1).values
    got = cm[:B, : ref.shape[1]]
    err = (got - ref).abs().max().item()
    assert err < 2e-3, f"chunkmax abs err {err}"
    rs = part.sum(0)[:B]
    rref = torch.exp(S - c[:B, None]).sum(1)
    assert ((rs - rref).abs() / rref).max().item() < 2e-3


@pytest.mark.parametrize("B,N", [(512, 5000), (200, 2333), (64, 40000)])
def test_score_bwd_q(native, B, N):
    g = torch.Generator(device="cuda").manual_seed(B + N)
    n_pad = (N + 255) // 256 * 256
    E = torch.zeros(QROWS, n_pad, device="cuda", dtype=torch.bfloat16)
    E[:B, :N] = torch.rand(B, N, device="cuda", generator=g).bfloat16()
    I = torch.zeros(n_pad, KEXT, device="cuda", dtype=torch.bfloat16)
    I[:N] = (torch.randn(N, KEXT, device="cuda", generator=g) * 0.1).bfloat16()
    splits = native.lib().tcar_score_bwd_q_splits(B, n_pad)
    part = torch.zeros(splits, QROWS, KEXT, device="cuda")
    dq = torch.zeros(QROWS, KEXT, device="cuda")
    native.call("tcar_score_bwd_q", native.ptr(e_to_blocked(E)), native.ptr(I), native.ptr(part), native.ptr(dq), B,
                n_pad)
    torch.cuda.synchronize()
    ref = (E[:B].double() @ I.double()).float()
    scale = ref.abs().max().item()
    err = (dq[:B] - ref).abs().max().item() / scale
    assert err < 1e-4, f"dq err {err} (scale {scale})"


@pytest.mark.parametrize("B,N", [(512, 5000), (200, 2333), (64, 40000), (5, 300)])
def test_score_bwd_i(native, B, N):
    g = torch.Generator(device="cuda").manual_seed(3 * B + N)
    n_pad = (N + 255) // 256 * 256
    kpad = (B + 63) // 64 * 64
    E = torch.zeros(QROWS, n_pad, device="cuda", dtype=torch.bfloat16)
    E[:B, :N] = torch.rand(B, N, device="cuda", generator=g).bfloat16()
    E[kpad:] = float("nan")  # rows beyond the K padding must never be read
    Qs = torch.zeros(QROWS, 256, device="cuda", dtype=torch.bfloat16)
    Qs[:B, :250] = (torch.randn(B, 250, device="cuda", generator=g) * 0.2).bfloat16()
    gi = torch.full((N + 1, 256), float("nan"), device="cuda")
    gi[0] = 0
    sqp = torch.full((native.lib().tcar_score_bwd_i_ctas(n_pad),), float("nan"), device="cuda")
    native.call("tcar_score_bwd_i", native.ptr(e_to_blocked(E)), native.ptr(Qs), native.ptr(gi), native.ptr(sqp), B, N,
                n_pad)
    torch.cuda.synchronize()
    ref = (E[:B, :N].double().t() @ Qs[:B].double()).float()
    scale = ref.abs().max().item()
    err = (gi[1:] - ref).abs().max().item() / scale
    assert err < 1e-4, f"g_item err {err} (scale {scale})"
    assert (gi[1:, 250:] == 0).all()
    assert (gi[0] == 0).all()
    # the fused per-CTA sums of squares add up to ||g_item||^2
    want = float((gi.double() ** 2).sum())
    assert abs(float(sqp.double().sum()) - want) <= 1e-5 * want


@pytest.mark.parametrize("B,N", [(512, 5000), (77, 2333)])
def test_score_bwd_i_tma_epilogue_equals_the_row_store_kernel(native, B, N):
    """The staged TMA-store epilogue (tcar_score_bwd_i) and the row-store kernel (thread <-> row stores; what
    tcar_score_bwd_i_acc runs with accumulate = 1, here into a zero gradient, where 0 + x is exact) run the same MMAs
    in the same order: gradient and per-CTA sums of squares bit-identical; rows beyond the table untouched."""
    g = torch.Generator(device="cuda").manual_seed(B + N)
    n_pad = (N + 255) // 256 * 256
    E = torch.zeros(QROWS, n_pad, device="cuda", dtype=torch.bfloat16)
    E[:B, :N] = torch.rand(B, N, device="cuda", generator=g).bfloat16()
    Qs = torch.zeros(QROWS, 256, device="cuda", dtype=torch.bfloat16)
    Qs[:B, :250] = (torch.randn(B, 250, device="cuda", generator=g) * 0.2).bfloat16()
    Eb = e_to_blocked(E)
    ctas = native.lib().tcar_score_bwd_i_ctas(n_pad)
    gi = torch.full((N + 1 + 300, 256), 7.0, device="cuda")              # 300 guard rows behind the table
    sqp = torch.zeros(ctas, device="cuda")
    native.call("tcar_score_bwd_i", native.ptr(Eb), native.ptr(Qs), native.ptr(gi), native.ptr(sqp), B, N, n_pad)
    ref = torch.zeros(N + 1, 256, device="cuda")
    ref_sqp = torch.zeros(ctas, device="cuda")
    native.call("tcar_score_bwd_i_acc", native.ptr(Eb), native.ptr(Qs), native.ptr(ref), native.ptr(ref_sqp), B, N,
                n_pad, 1)
    torch.cuda.synchronize()
    assert torch.equal(gi[1: N + 1], ref[1:])
    assert torch.equal(sqp, ref_sqp)
    assert (gi[0] == 7.0).all() and (gi[N + 1:] == 7.0).all()


# ------------------------------------------------------------------------------------------- session groups (catalog-sharded step)
@pytest.mark.parametrize("counts,N", [([512, 512], 5000), ([300, 0, 512, 77], 2333), ([512] * 8, 3000), ([1, 5], 300)])
def test_score_groups_match_single_group_calls(native, counts, N):
    """tcar_score_fwd_groups / _bwd_q_groups (one launch over all groups, tcar_score_bwd_q_multi) / _bwd_i_groups
    against the per-group entry points and a torch matmul over the same bf16 operands."""
    R = len(counts)
    g = torch.Generator(device="cuda").manual_seed(N + R)
    n_pad = (N + 255) // 256 * 256
    lib = native.lib()
    tiles = lib.tcar_score_fwd_tiles(n_pad)
    I = torch.zeros(n_pad, KEXT, device="cuda", dtype=torch.bfloat16)
    I[:N] = (torch.randn(N, KEXT, device="cuda", generator=g) * 0.1).bfloat16()
    I[:, KEXT - 1] = 0                                # the pad column of the scoring operand is zero
    Q = torch.zeros(R, QROWS, KEXT, device="cuda", dtype=torch.bfloat16)
    c = torch.randn(R, QROWS, device="cuda", generator=g) * 0.3
    for r, b in enumerate(counts):
        Q[r, :b] = (torch.randn(b, KEXT, device="cuda", generator=g) * 0.5).bfloat16()
    E = torch.zeros(R, QROWS * n_pad, device="cuda", dtype=torch.bfloat16)
    part = torch.zeros(R, tiles * QROWS, device="cuda")
    cnt = (C.c_int * R)(*counts)
    p = native.ptr
    native.call("tcar_score_fwd_groups", p(Q), QROWS * KEXT, p(c), QROWS, p(I), p(E), QROWS * n_pad, p(part),
                tiles * QROWS, cnt, R, N, n_pad, -2)
    torch.cuda.synchronize()
    for r, b in enumerate(counts):
        if b == 0:
            assert (E[r] == 0).all()
            continue
        E1 = torch.zeros(QROWS, n_pad, device="cuda", dtype=torch.bfloat16)
        p1 = torch.zeros(tiles, QROWS, device="cuda")
        native.call("tcar_score_fwd", p(Q[r]), p(I), p(c[r]), p(E1), p(p1), None, None, b, N, n_pad, 0, -2)
        torch.cuda.synchronize()
        assert torch.equal(E1.view(-1), E[r]) and torch.equal(p1.view(-1)[: tiles * QROWS], part[r])
    # ---- dQ: tcar_score_bwd_q_groups (one launch over all groups when several are present) vs per-group
    # tcar_score_bwd_q + tcar_rowsum_finish calls vs fp64 matmul
    qelems = max(int(lib.tcar_score_bwd_q_multi_part_elems(R)),
                 max(lib.tcar_score_bwd_q_splits(b, n_pad) for b in (1, 129, 257, 385)) * QROWS * KEXT)
    qpart = torch.zeros(qelems, device="cuda")
    dq = torch.zeros(R, QROWS, KEXT, device="cuda")
    native.call("tcar_score_bwd_q_groups", p(E), QROWS * n_pad, p(I), p(qpart), p(dq), QROWS * KEXT, p(part),
                tiles * QROWS, tiles, cnt, R, n_pad)
    torch.cuda.synchronize()
    for r, b in enumerate(counts):
        if b == 0:
            continue
        dq1 = torch.zeros(QROWS, KEXT, device="cuda")
        native.call("tcar_score_bwd_q", p(E[r]), p(I), p(qpart), p(dq1), b, n_pad)
        native.call("tcar_rowsum_finish", p(part[r]), p(dq1[:, KEXT - 1:]), KEXT, tiles, b)
        torch.cuda.synchronize()
        El = e_from_blocked(E[r], n_pad)[:b].double()
        ref = (El @ I.double()).float()
        ref[:, KEXT - 1] = El.float().sum(1)          # softmax partial sums ride in the pad column
        scale = ref[:, : KEXT - 1].abs().max().item()
        for name, got in (("groups", dq[r, :b]), ("single", dq1[:b])):
            assert (got[:, : KEXT - 1] - ref[:, : KEXT - 1]).abs().max().item() / scale < 1e-4, (name, r)
            rs = got[:, KEXT - 1]
            assert ((rs - ref[:, KEXT - 1]).abs() / ref[:, KEXT - 1]).max().item() < 2e-3, (name, r)
        assert torch.equal(dq[r, :b, KEXT - 1], dq1[:b, KEXT - 1])
    # ---- dItems: first present group overwrites, later ones accumulate
    Qs = torch.zeros(R, QROWS, 256, device="cuda", dtype=torch.bfloat16)
    for r, b in enumerate(counts):
        Qs[r, :b, :250] = (torch.randn(b, 250, device="cuda", generator=g) * 0.2).bfloat16()
    gi = torch.full((N + 1, 256), float("nan"), device="cuda")
    gi[0] = 0
    sqp = torch.zeros(lib.tcar_score_bwd_i_ctas(n_pad), device="cuda")
    native.call("tcar_score_bwd_i_groups", p(E), QROWS * n_pad, p(Qs), QROWS * 256, p(gi), p(sqp), cnt, R, N, n_pad)
    torch.cuda.synchronize()
    ref = sum(e_from_blocked(E[r], n_pad)[:b, :N].double().t() @ Qs[r, :b].double() for r, b in enumerate(counts) if b)
    scale = ref.abs().max().item()
    assert (gi[1:].double() - ref).abs().max().item() / scale < 1e-4
    want = float((gi.double() ** 2).sum())
    assert abs(float(sqp.double().sum()) - want) <= 1e-5 * want


@pytest.mark.parametrize("counts,N", [([512, 200, 512], 4000), ([77, 512], 1500)])
def test_score_groups_overflow_guard_matches_single_group_calls(native, counts, N):
    """Both passes of the softmax overflow guard over several session groups in one launch each
    (tcar_score_fwd_groups_guarded -> score_fwd_multi_kernel, tcar_rowmax_groups) against the single-group entry points:
    E, partial sums and row maxima bit-identical; rows whose label score lies ~200 nats below their best candidate get
    the extra shift (finite E, largest term 2^0), quiet rows keep their pass-1 values."""
    R = len(counts)
    g = torch.Generator(device="cuda").manual_seed(N + R)
    n_pad = (N + 255) // 256 * 256
    lib = native.lib()
    tiles = lib.tcar_score_fwd_tiles(n_pad)
    I = torch.zeros(n_pad, KEXT, device="cuda", dtype=torch.bfloat16)
    I[:N] = (torch.randn(N, KEXT, device="cuda", generator=g) * 0.1).bfloat16()
    Q = torch.zeros(R, QROWS, KEXT, device="cuda", dtype=torch.bfloat16)
    c = torch.randn(R, QROWS, device="cuda", generator=g) * 0.3
    for r, b in enumerate(counts):
        Q[r, :b] = (torch.randn(b, KEXT, device="cuda", generator=g) * 0.5).bfloat16()
        c[r, 3:b:37] -= 200.0                      # these rows overflow exp(S - c) without the guard
    E = torch.zeros(R, QROWS * n_pad, device="cuda", dtype=torch.bfloat16)
    part = torch.zeros(R, tiles * QROWS, device="cuda")
    pmax = torch.zeros(R, tiles * QROWS, device="cuda")
    rowmax = torch.zeros(R, QROWS, device="cuda")
    cnt = (C.c_int * R)(*counts)
    p = native.ptr
    args = (p(Q), QROWS * KEXT, p(c), QROWS, p(I), p(E), QROWS * n_pad, p(part), tiles * QROWS)
    native.call("tcar_score_fwd_groups_guarded", *args, p(pmax), None, cnt, R, N, n_pad, -2)
    native.call("tcar_rowmax_groups", p(pmax), tiles * QROWS, p(rowmax), tiles, cnt, R)
    torch.cuda.synchronize()
    E_pass1 = E.clone()
    native.call("tcar_score_fwd_groups_guarded", *args, None, p(rowmax), cnt, R, N, n_pad, -2)
    torch.cuda.synchronize()
    assert torch.isfinite(E.float()).all() and torch.isfinite(part).all()
    for r, b in enumerate(counts):
        E1 = torch.zeros(QROWS, n_pad, device="cuda", dtype=torch.bfloat16)
        p1 = torch.zeros(tiles, QROWS, device="cuda")
        m1 = torch.zeros(tiles, QROWS, device="cuda")
        rm1 = torch.zeros(QROWS, device="cuda")
        se, ce = torch.zeros(QROWS, device="cuda"), torch.zeros(QROWS, device="cuda")
        native.call("tcar_score_fwd_guarded", p(Q[r]), p(I), p(c[r]), p(E1), p(p1), None, None, p(m1), None, b, N, n_pad, 0, -2)
        native.call("tcar_ce_finish_guarded", p(p1), p(m1), p(se), p(ce), p(rm1), tiles, b, 1)
        torch.cuda.synchronize()
        assert torch.equal(m1.view(-1), pmax[r]) and torch.equal(rm1[:b], rowmax[r, :b])
        hot = rm1[:b] > 80.0
        assert int(hot.sum()) == len(range(3, b, 37)) and bool(hot[3])
        native.call("tcar_score_fwd_guarded", p(Q[r]), p(I), p(c[r]), p(E1), p(p1), None, None, None, p(rm1), b, N, n_pad, 0, -2)
        native.call("tcar_ce_finish_guarded", p(p1), None, p(se), p(ce), p(rm1), tiles, b, 2)
        torch.cuda.synchronize()
        assert torch.equal(E1.view(-1), E[r]) and torch.equal(p1.view(-1), part[r])
        # CE of a shifted row = logsumexp(S) - c, against fp64 over the same bf16 operands
        S = Q[r, :b].double() @ I[:N].double().t()
        want = torch.logsumexp(S, 1) - c[r, :b].double()
        np.testing.assert_allclose(ce[:b].cpu().double().numpy(), want.cpu().numpy(), rtol=2e-5, atol=2e-4)
        # quiet rows: pass 2 left their E untouched
        Eb1 = E_pass1[r].view(n_pad // 8, QROWS, 8)
        Eb2 = E[r].view(n_pad // 8, QROWS, 8)
        quiet = (~hot).nonzero().flatten()
        assert torch.equal(Eb1[:, quiet], Eb2[:, quiet])
