"""GPU parity tests (run with `-m gpu` on a B200). Everything goes through the public API -> C ABI -> CUDA kernels and
is checked against the CPU oracle (oracle/blockwise.py) on seeded inputs, against committed golden fixtures produced
by the reference's own SM100 kernel (tests/golden/gpu_golden.*.pt), and -- at BASELINE.json's full sizes -- through
size-independent properties (linearity in the power-of-two scales, row/column permutation equivariance, zero rows).

Tolerance: every e4m3 x e4m3 product and every UE8M0 scale is exact, so the only freedom versus the oracle is the
FP32 accumulation order inside the tensor core. FP32 outputs: |d - oracle| <= 1e-5 * max|oracle| (a handful of FP32
roundings of the accumulator); BF16 outputs: differ on at most 1% of the elements, each by at most one BF16 rounding
step of the value plus that FP32 noise, and calc_diff < 1e-6 (the reference's own
test bound is 1e-3 against unquantised inputs, tests/test_fp8_fp4.py:53-55). Versus the reference's SM100 kernel on
identical inputs the match is BITWISE (golden fixtures).
"""
import os
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope='module')
def dg():
    if not torch.cuda.is_available():
        pytest.skip('needs a GPU')
    import deepgemm_b200
    from deepgemm_b200 import _lib
    _lib.lib()  # fail loudly if the CUDA library is missing: there is no fallback
    return deepgemm_b200


def _quant_dense(m, n, k, seed=0):
    from deepgemm_b200.utils import per_block_cast_to_fp8, per_token_cast_to_fp8
    g = torch.Generator(device='cuda').manual_seed(seed)
    a = torch.randn((m, k), device='cuda', dtype=torch.bfloat16, generator=g)
    b = torch.randn((n, k), device='cuda', dtype=torch.bfloat16, generator=g)
    return a, b, per_token_cast_to_fp8(a, True), per_block_cast_to_fp8(b, True)


def _cpu(pair):
    return pair[0].cpu(), pair[1].cpu()


def _assert_close_to_oracle(d, want, what='', mag=None):
    """`mag`: magnitude that sets the BF16 rounding step (defaults to |want|; with C accumulation the product is rounded
    to BF16 BEFORE the add, so the step is that of |product| + |C|, not of the possibly cancelled sum)."""
    from deepgemm_b200.testing import calc_diff
    d, want = d.cpu(), want.cpu()
    mag = want.float().abs() if mag is None else mag.cpu().float()
    assert d.shape == want.shape, what
    if d.numel() == 0:
        return
    assert not torch.isnan(d.float()).any(), what
    assert calc_diff(d, want) < 1e-6, what
    if d.dtype == torch.bfloat16:
        mism = d != want
        assert mism.float().mean() <= 0.02, f'{what}: {int(mism.sum())} mismatches'
        # a mismatch is one BF16 rounding step of the value (2^-7 relative) plus FP32 accumulation noise, which is
        # absolute (it scales with sum_k |a_k b_k|, not with the possibly cancelled result)
        err = (d.float() - want.float()).abs()
        tol = mag * 2.0 ** -7 + 1e-5 * mag.max()
        assert bool((err <= tol).all()), f'{what}: max excess {float((err - tol).max())}'
    else:
        scale = want.abs().max().clamp(min=1.0)
        assert ((d - want).abs().max() / scale) < 1e-5, what


@pytest.mark.parametrize('m,n,k', [(128, 128, 128), (1, 576, 512), (64, 4096, 7168), (300, 2112, 1536), (257, 384, 7296),
                                   (96, 130, 200)])
@pytest.mark.parametrize('out_dtype', [torch.bfloat16, torch.float32])
def test_dense_matches_oracle(dg, m, n, k, out_dtype):
    from oracle import blockwise
    if k % 16:
        pytest.skip('TMA needs 16-byte rows')
    a, b, qa, qb = _quant_dense(m, n, k, seed=m + n + k)
    d = torch.full((m, n), float('nan'), device='cuda', dtype=out_dtype)
    dg.fp8_gemm_nt(qa, qb, d)
    want = blockwise.fp8_gemm_nt(_cpu(qa), _cpu(qb), out_dtype=out_dtype)
    _assert_close_to_oracle(d, want, f'{m}x{n}x{k}')
    # the reference's own tolerance against the unquantised product
    from deepgemm_b200.testing import calc_diff
    assert calc_diff(d, a.float() @ b.float().t()) < 1e-3


@pytest.mark.parametrize('cfg', [(16, 1, 2), (32, 2, 3), (64, 2, 0), (112, 1, 4), (128, 2, 0), (240, 2, 0), (208, 1, 0)])
def test_dense_every_tile_config_gives_identical_bits(dg, cfg, monkeypatch):
    """Tile height / CTA pairing / pipeline depth are performance knobs only: FP32 accumulation runs over K in the
    same order whatever the tile shape, so the output bits must not depend on them."""
    m, n, k = 500, 1024, 2048
    _, _, qa, qb = _quant_dense(m, n, k, seed=7)
    base = torch.empty((m, n), device='cuda', dtype=torch.bfloat16)
    monkeypatch.setenv('DGB200_SPLITS', '1')     # split-K (small problems) changes the FP32 summation order
    dg.fp8_gemm_nt(qa, qb, base)
    bm, cl, st = cfg
    monkeypatch.setenv('DGB200_BLOCK_M', str(bm))
    monkeypatch.setenv('DGB200_CLUSTER', str(cl))
    if st:
        monkeypatch.setenv('DGB200_STAGES', str(st))
    d = torch.empty_like(base)
    dg.fp8_gemm_nt(qa, qb, d)
    from deepgemm_b200 import _lib
    assert _lib.last_config()['block_m'] == bm and _lib.last_config()['cluster'] == cl
    assert torch.equal(d, base)


@pytest.mark.parametrize('m,n,k,splits', [(64, 4096, 7168, 4), (128, 1024, 2048, 4), (200, 768, 7168, 8), (1, 2112, 7168, 0),
                                          (96, 512, 1664, 3)])
@pytest.mark.parametrize('out_dtype', [torch.bfloat16, torch.float32])
def test_dense_split_k_matches_oracle_and_is_deterministic(dg, m, n, k, splits, out_dtype, monkeypatch):
    """Small problems cut K into slices (every SM streams its own part of B); partial sums are added in slice order."""
    from deepgemm_b200 import _lib
    from oracle import blockwise
    _, _, qa, qb = _quant_dense(m, n, k, seed=m + k)
    if splits:
        monkeypatch.setenv('DGB200_SPLITS', str(splits))
    outs = []
    for _ in range(3):
        d = torch.full((m, n), float('nan'), device='cuda', dtype=out_dtype)
        dg.fp8_gemm_nt(qa, qb, d)
        outs.append(d)
    assert _lib.last_config()['num_splits'] > 1, _lib.last_config()
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])     # run-to-run deterministic
    _assert_close_to_oracle(outs[0], blockwise.fp8_gemm_nt(_cpu(qa), _cpu(qb), out_dtype=out_dtype), f'split-k {m}x{n}x{k}')
    # accumulation into C goes through the same finalising pass
    c = (torch.randn((m, n), device='cuda', generator=torch.Generator(device='cuda').manual_seed(m + n)) * 8).to(out_dtype)
    d = c.clone()
    dg.fp8_gemm_nt(qa, qb, d, c=d)
    # three BF16 roundings separate the two results (kernel: product, then sum; oracle: sum), each half a step of its
    # operand: |err| <= 2^-8 (|prod| + 2 |prod + c|) <= 1.5 * 2^-7 (|prod| + |c|)
    _assert_close_to_oracle(d, blockwise.fp8_gemm_nt(_cpu(qa), _cpu(qb), out_dtype=out_dtype, c=c.cpu()), 'split-k + C',
                            mag=1.5 * (outs[0].float().abs() + c.float().abs()))
    # and without slices the kernel still agrees (different summation order: tolerance, not bits)
    monkeypatch.setenv('DGB200_SPLITS', '1')
    d1 = torch.empty((m, n), device='cuda', dtype=out_dtype)
    dg.fp8_gemm_nt(qa, qb, d1)
    assert _lib.last_config()['num_splits'] == 1
    _assert_close_to_oracle(outs[0], d1, 'split vs unsplit')


@pytest.mark.parametrize('m,n,k,cs', [(64, 4096, 7168, 4), (128, 4096, 7168, 4), (1, 2112, 7168, 4), (100, 520, 1536, 4),
                                      (64, 1024, 512, 2), (200, 384, 2048, 2), (33, 136, 1408, 2)])
@pytest.mark.parametrize('out_dtype', [torch.bfloat16, torch.float32])
def test_dense_cluster_split_k_matches_oracle_and_is_deterministic(dg, m, n, k, cs, out_dtype, monkeypatch):
    """Split-K inside a cluster: `cs` single-CTA MMAs each accumulate one K slice of the same output tile and exchange
    the partial tiles through distributed shared memory (csrc/fp8_gemm_kernel.cuh, kCSplit). Slices are added in a
    fixed order: deterministic, equal to the oracle to FP32 rounding; set_split_k(False) restores the one-pass bits."""
    from deepgemm_b200 import _lib
    from oracle import blockwise
    _, _, qa, qb = _quant_dense(m, n, k, seed=m + n)
    monkeypatch.setenv('DGB200_CSPLIT', str(cs))
    outs = []
    for _ in range(3):
        d = torch.full((m, n), float('nan'), device='cuda', dtype=out_dtype)
        dg.fp8_gemm_nt(qa, qb, d)
        outs.append(d)
    cfg = _lib.last_config()
    assert cfg['cluster_split'] == cs and cfg['cluster'] == cs and cfg['num_splits'] == cs, cfg
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    want = blockwise.fp8_gemm_nt(_cpu(qa), _cpu(qb), out_dtype=out_dtype)
    _assert_close_to_oracle(outs[0], want, f'cluster split-k {m}x{n}x{k}')
    # accumulate into C
    c = (torch.randn((m, n), device='cuda', generator=torch.Generator(device='cuda').manual_seed(m + k)) * 8).to(out_dtype)
    d = c.clone()
    dg.fp8_gemm_nt(qa, qb, d, c=d)
    _assert_close_to_oracle(d, blockwise.fp8_gemm_nt(_cpu(qa), _cpu(qb), out_dtype=out_dtype, c=c.cpu()), 'cluster split-k + C',
                            mag=1.5 * (outs[0].float().abs() + c.float().abs()))
    # the knob: no split -> same bits as the single-pass kernel
    monkeypatch.delenv('DGB200_CSPLIT')
    dg.set_split_k(False)
    try:
        d1 = torch.empty((m, n), device='cuda', dtype=out_dtype)
        dg.fp8_gemm_nt(qa, qb, d1)
        assert _lib.last_config()['num_splits'] == 1 and _lib.last_config()['cluster_split'] == 0
    finally:
        dg.set_split_k(True)
    monkeypatch.setenv('DGB200_SPLITS', '1')
    d2 = torch.empty((m, n), device='cuda', dtype=out_dtype)
    dg.fp8_gemm_nt(qa, qb, d2)
    assert torch.equal(d1, d2)
    _assert_close_to_oracle(outs[0], d1, 'split vs unsplit')


@pytest.mark.parametrize('m,n,k', [(4096, 4096, 512), (2000, 2112, 640), (1024, 7168, 256), (3333, 512, 384)])
def test_dense_wave_balanced_tile_heights_give_identical_bits(dg, m, n, k, monkeypatch):
    """Large dense problems pick the NUMBER of m-blocks that fills whole rounds of CTA pairs and use two tile heights
    (block_m and block_m - 16). Heights are a scheduling matter only: same bits as uniform tiles."""
    from deepgemm_b200 import _lib
    _, _, qa, qb = _quant_dense(m, n, k, seed=k)
    monkeypatch.setenv('DGB200_BALANCE', '0')
    base = torch.empty((m, n), device='cuda', dtype=torch.bfloat16)
    dg.fp8_gemm_nt(qa, qb, base)
    uniform = _lib.last_config()
    monkeypatch.setenv('DGB200_BALANCE', '1')
    d = torch.full((m, n), float('nan'), device='cuda', dtype=torch.bfloat16)
    dg.fp8_gemm_nt(qa, qb, d)
    assert torch.equal(d, base), (uniform, _lib.last_config())
    c = torch.randn((m, n), device='cuda', generator=torch.Generator(device='cuda').manual_seed(1)).to(torch.bfloat16)
    d1, d2 = c.clone(), c.clone()
    dg.fp8_gemm_nt(qa, qb, d1, c=d1)
    monkeypatch.setenv('DGB200_BALANCE', '0')
    dg.fp8_gemm_nt(qa, qb, d2, c=d2)
    assert torch.equal(d1, d2)


@pytest.mark.parametrize('out_dtype', [torch.bfloat16, torch.float32])
def test_dense_accumulate_into_c(dg, out_dtype):
    from oracle import blockwise
    m, n, k = 200, 512, 1024
    _, _, qa, qb = _quant_dense(m, n, k, seed=3)
    c = (torch.randn((m, n), device='cuda', generator=torch.Generator(device='cuda').manual_seed(11)) * 32).to(out_dtype)
    # c is d (in place)
    d = c.clone()
    dg.fp8_gemm_nt(qa, qb, d, c=d)
    want = blockwise.fp8_gemm_nt(_cpu(qa), _cpu(qb), out_dtype=out_dtype, c=c.cpu())
    _assert_close_to_oracle(d, want, 'in-place accumulate',
                            mag=1.5 * ((want.float() - c.cpu().float()).abs() + c.cpu().float().abs()))
    # c separate from d: d <- c first (csrc/apis/gemm.hpp:42-44), c untouched
    d2 = torch.empty_like(c)
    c_before = c.clone()
    dg.fp8_gemm_nt(qa, qb, d2, c=c)
    assert torch.equal(d2, d) and torch.equal(c, c_before)


def test_dense_packed_int_sf_inputs_equal_fp32_sf_inputs(dg):
    """Callers may pass pre-packed UE8M0 int32 scale factors in the documented layout (csrc/apis/layout.hpp:56-58)."""
    m, n, k = 130, 256, 1536
    _, _, qa, qb = _quant_dense(m, n, k, seed=11)
    d0 = torch.empty((m, n), device='cuda', dtype=torch.bfloat16)
    dg.fp8_gemm_nt(qa, qb, d0)
    sfa = dg.transform_sf_into_required_layout(qa[1], m, k, (1, 128, 128), None, True)
    sfb = dg.transform_sf_into_required_layout(qb[1], n, k, (1, 128, 128), None, False)
    assert sfa.dtype == torch.int32 and sfa.shape == (m, 3) and sfa.stride() == (1, 132)
    d1 = torch.empty_like(d0)
    dg.fp8_gemm_nt((qa[0], sfa), (qb[0], sfb), d1)          # default recipe for int SFs is (1, 1, 128)
    assert torch.equal(d0, d1)
    d2 = torch.empty_like(d0)
    dg.fp8_gemm_nt((qa[0], sfa), (qb[0], sfb), d2, recipe_a=(1, 128), recipe_b=(1, 128))
    assert torch.equal(d0, d2)


def test_sf_pack_kernel_bit_exact(dg):
    """The reference pins these kernels bit-exactly (tests/test_layout.py:58-60): shape, strides and bytes."""
    from deepgemm_b200.utils import per_token_cast_to_fp8
    from oracle import blockwise
    for mn, k, groups, gran_k in [(4096, 7168, 1, 128), (4097, 7296, 1, 128), (130, 128, 4, 128), (513, 384, 2, 32),
                                  (8192, 7168, 2, 128)]:
        x = torch.randn((groups * mn, k), device='cuda', dtype=torch.bfloat16)
        _, sf = per_token_cast_to_fp8(x, True, gran_k)
        sf = sf if groups == 1 else sf.view(groups, mn, -1)
        for transposed_input in (False, True):
            src = sf.transpose(-1, -2).contiguous().transpose(-1, -2) if transposed_input else sf
            packed = dg.get_mn_major_tma_aligned_packed_ue8m0_tensor(src)
            want = blockwise.pack_sf_ue8m0_mn_major(sf.cpu())
            assert packed.shape == want.shape and packed.stride() == want.stride()
            assert torch.equal(packed.cpu(), want), (mn, k, groups, transposed_input)
    # FP32 MN-major utility
    sf = torch.rand((3, 100, 7), device='cuda')
    t = dg.get_mn_major_tma_aligned_tensor(sf)
    assert t.shape == sf.shape and t.stride() == (7 * 100, 1, 100) and torch.equal(t, sf)


@pytest.mark.parametrize('layout', ['nn', 'tn', 'tt'])
@pytest.mark.parametrize('m,n,k', [(256, 384, 512), (4096, 512, 1024), (192, 2112, 1536), (112, 256, 640)])
def test_dense_layout_variants_match_nt_bitwise(dg, layout, m, n, k):
    """fp8_gemm_{nn,tn,tt}: MN-major operands (csrc/apis/gemm.hpp:126-164). Same numbers, same K order as the NT call on
    the same quantised data, so the outputs must be bit-identical to it (and NT is pinned to the oracle above)."""
    _, _, qa, qb = _quant_dense(m, n, k, seed=k)
    d_nt = torch.empty((m, n), device='cuda', dtype=torch.bfloat16)
    dg.fp8_gemm_nt(qa, qb, d_nt)
    a_t = (qa[0].t().contiguous(), qa[1].t().contiguous())       # A given as [K, M]
    b_t = (qb[0].t().contiguous(), qb[1].t().contiguous())       # B given as [K, N]
    d = torch.full((m, n), float('nan'), device='cuda', dtype=torch.bfloat16)
    if layout == 'nn':
        dg.fp8_gemm_nn(qa, b_t, d)
    elif layout == 'tn':
        dg.fp8_gemm_tn(a_t, b_t, d)
    else:
        dg.fp8_gemm_tt(a_t, qb, d)
    assert torch.equal(d, d_nt), layout


@pytest.mark.parametrize('gran_k', [128, 32])
@pytest.mark.parametrize('use_psum', [False, True])
def test_k_grouped_matches_oracle(dg, gran_k, use_psum):
    """Weight gradient: D[g] = C[g] + A_g^T B_g, FP32 in place (tests/test_fp8_fp4.py:193-242 covers the same cases:
    empty groups, K tails, gran_k 32/128, psum layout with unaligned group ends)."""
    from deepgemm_b200.utils import per_channel_cast_to_fp8
    from oracle import blockwise
    random.seed(gran_k + use_psum)
    gen = torch.Generator(device='cuda').manual_seed(9)
    g, m, n = 5, 512, 384
    k_alignment = 128 if gran_k == 128 else 32
    dg.set_mk_alignment_for_contiguous_layout(k_alignment)
    try:
        real_ks = [k_alignment * random.randint(1, 6) for _ in range(g)]
        real_ks[1] = 0                                              # an empty group
        real_ks[3] = k_alignment                                    # a K tail shorter than one k-block (when 32)
        if use_psum:
            real_ks[0] -= 7                                         # psum: group ends need not be aligned
            ends, prev = [], 0
            for kk in real_ks:
                prev = blockwise.align(prev, k_alignment) + kk
                ends.append(prev)
            total_k = blockwise.align(ends[-1], k_alignment)
        else:
            ends, total_k = None, sum(real_ks)
        a = torch.zeros((total_k, m), device='cuda', dtype=torch.bfloat16)
        b = torch.zeros((total_k, n), device='cuda', dtype=torch.bfloat16)
        a8 = torch.zeros((total_k, m), device='cuda', dtype=torch.float8_e4m3fn)
        b8 = torch.zeros((total_k, n), device='cuda', dtype=torch.float8_e4m3fn)
        sfa_l, sfb_l, pos = [], [], 0
        for i, kk in enumerate(real_ks):
            end = ends[i] if use_psum else pos + kk
            start = end - kk
            pos = end
            if kk == 0:
                continue
            pad = blockwise.align(kk, gran_k)
            xa = torch.zeros((pad, m), device='cuda', dtype=torch.bfloat16)
            xb = torch.zeros((pad, n), device='cuda', dtype=torch.bfloat16)
            xa[:kk] = torch.randn((kk, m), device='cuda', dtype=torch.bfloat16, generator=gen)
            xb[:kk] = torch.randn((kk, n), device='cuda', dtype=torch.bfloat16, generator=gen)
            qa, sa = per_channel_cast_to_fp8(xa, True, gran_k)
            qb, sb = per_channel_cast_to_fp8(xb, True, gran_k)
            a8[start:end], b8[start:end] = qa[:kk], qb[:kk]
            sfa_l.append(sa), sfb_l.append(sb)
        sfa, sfb = torch.cat(sfa_l), torch.cat(sfb_l)
        c = torch.randn((g, m, n), device='cuda', generator=gen) * 32
        d = c.clone()
        layout = torch.tensor(ends if use_psum else real_ks, device='cuda', dtype=torch.int32)
        ks_arg = [blockwise.align(kk, k_alignment) for kk in real_ks] if use_psum else real_ks
        dg.k_grouped_fp8_gemm_tn_contiguous((a8, sfa), (b8, sfb), d, ks_arg, layout, c=d, recipe=(1, 1, gran_k),
                                            use_psum_layout=use_psum)
        want = blockwise.k_grouped_fp8_gemm_tn_contiguous((a8.cpu(), sfa.cpu()), (b8.cpu(), sfb.cpu()), c.cpu(), real_ks, gran_k,
                                                          group_ends=ends)
        _assert_close_to_oracle(d, want, f'k-grouped gran_k={gran_k} psum={use_psum}')
        assert torch.equal(d[1], c[1])                              # the empty group left its D block untouched
        if not use_psum:
            packed = dg.get_k_grouped_mn_major_tma_aligned_packed_ue8m0_tensor(sfa, layout, real_ks, gran_k, k_alignment)
            assert torch.equal(packed.cpu(), blockwise.pack_sf_ue8m0_k_grouped(sfa.cpu(), real_ks, gran_k))
    finally:
        dg.set_mk_alignment_for_contiguous_layout(128)


def test_m_grouped_contiguous_nn_layout(dg):
    """m_grouped_fp8_gemm_nn_contiguous: B given as [G, K, N] (gemm.hpp:234-248) -- bit-identical to the NT call."""
    from deepgemm_b200.utils import per_token_cast_to_fp8
    gen = torch.Generator(device='cuda').manual_seed(12)
    g, n, k, per = 3, 512, 768, 128
    a = torch.randn((g * per, k), device='cuda', dtype=torch.bfloat16, generator=gen)
    qa = per_token_cast_to_fp8(a, True)
    _, qb = _grouped_weights(g, n, k, gen)
    layout = torch.arange(g, device='cuda', dtype=torch.int32).repeat_interleave(per)
    d_nt = torch.empty((g * per, n), device='cuda', dtype=torch.bfloat16)
    dg.m_grouped_fp8_gemm_nt_contiguous(qa, qb, d_nt, layout)
    b_kn = (qb[0].transpose(1, 2).contiguous(), qb[1].transpose(1, 2).contiguous())   # [G, K, N]
    d_nn = torch.full_like(d_nt, float('nan'))
    dg.m_grouped_fp8_gemm_nn_contiguous(qa, b_kn, d_nn, layout)
    assert torch.equal(d_nn, d_nt)


def _grouped_weights(g, n, k, gen):
    from deepgemm_b200.utils import per_block_cast_to_fp8
    b = torch.randn((g, n, k), device='cuda', dtype=torch.bfloat16, generator=gen)
    q = [per_block_cast_to_fp8(b[i], True) for i in range(g)]
    return b, (torch.stack([x[0] for x in q]), torch.stack([x[1] for x in q]))


@pytest.mark.parametrize('alignment', [128, 224, 64])
@pytest.mark.parametrize('use_psum', [False, True])
def test_m_grouped_contiguous_matches_oracle(dg, alignment, use_psum):
    from deepgemm_b200.utils import per_token_cast_to_fp8
    from oracle import blockwise
    random.seed(alignment + use_psum)
    gen = torch.Generator(device='cuda').manual_seed(5)
    g, n, k = 6, 768, 1024
    dg.set_mk_alignment_for_contiguous_layout(alignment)
    try:
        ms = [int(150 * random.uniform(0.3, 1.7)) for _ in range(g)]
        ms[2] = 0                                             # an expert without tokens
        aligned = [blockwise.align(x, alignment) for x in ms]
        m = sum(aligned)
        a = torch.randn((m, k), device='cuda', dtype=torch.bfloat16, generator=gen)
        layout = torch.empty(g if use_psum else m, device='cuda', dtype=torch.int32)
        start = 0
        for i, (mi, ai) in enumerate(zip(ms, aligned)):
            if use_psum:
                layout[i] = start + mi
            else:
                layout[start:start + mi] = i
                layout[start + mi:start + ai] = -1
            a[start + mi:start + ai] = 0
            start += ai
        _, qb = _grouped_weights(g, n, k, gen)
        qa = per_token_cast_to_fp8(a, True)
        d = torch.full((m, n), float('nan'), device='cuda', dtype=torch.bfloat16)
        dg.m_grouped_fp8_gemm_nt_contiguous(qa, qb, d, layout, use_psum_layout=use_psum)
        want, valid = blockwise.m_grouped_fp8_gemm_nt_contiguous(_cpu(qa), _cpu(qb), layout.cpu(), use_psum_layout=use_psum,
                                                                alignment=alignment)
        _assert_close_to_oracle(d.cpu()[valid], want[valid], f'contiguous a={alignment} psum={use_psum}')
        if use_psum:
            # ensure_zero_padding (default): gap rows of D are exactly zero (tests/test_fp8_fp4.py:22-29)
            assert torch.equal(d.cpu()[~valid], torch.zeros_like(d.cpu()[~valid]))
    finally:
        dg.set_mk_alignment_for_contiguous_layout(128)


@pytest.mark.parametrize('expected_m', [20, 100])
def test_m_grouped_masked_matches_oracle_and_leaves_invalid_rows_alone(dg, expected_m):
    from deepgemm_b200.utils import per_token_cast_to_fp8
    from oracle import blockwise
    random.seed(expected_m)
    gen = torch.Generator(device='cuda').manual_seed(6)
    g, m_max, n, k = 8, 192, 512, 1024
    a = torch.randn((g, m_max, k), device='cuda', dtype=torch.bfloat16, generator=gen)
    q = [per_token_cast_to_fp8(a[i], True) for i in range(g)]
    qa = (torch.stack([x[0] for x in q]), torch.stack([x[1] for x in q]))
    _, qb = _grouped_weights(g, n, k, gen)
    masked_m = torch.tensor([min(m_max, int(expected_m * random.uniform(0.7, 1.3))) for _ in range(g)], device='cuda',
                            dtype=torch.int32)
    masked_m[3] = 0
    sentinel = 1234.0
    d = torch.full((g, m_max, n), sentinel, device='cuda', dtype=torch.bfloat16)
    dg.m_grouped_fp8_gemm_nt_masked(qa, qb, d, masked_m, expected_m)
    want = blockwise.m_grouped_fp8_gemm_nt_masked(_cpu(qa), _cpu(qb), masked_m.cpu())
    for gi, mg in enumerate(masked_m.tolist()):
        _assert_close_to_oracle(d[gi, :mg], want[gi, :mg], f'masked group {gi}')
        assert bool((d[gi, mg:] == sentinel).all()), 'rows >= masked_m must not be written'


def test_masked_is_cuda_graph_capturable(dg):
    """Config 4 runs under a CUDA graph: no host read of `masked_m`, no sync, no allocation with pre-packed SFs."""
    from deepgemm_b200.utils import per_token_cast_to_fp8
    gen = torch.Generator(device='cuda').manual_seed(8)
    g, m_max, n, k = 4, 128, 256, 512
    a = torch.randn((g, m_max, k), device='cuda', dtype=torch.bfloat16, generator=gen)
    q = [per_token_cast_to_fp8(a[i], True) for i in range(g)]
    qa = (torch.stack([x[0] for x in q]), torch.stack([x[1] for x in q]))
    _, qb = _grouped_weights(g, n, k, gen)
    sfa = dg.transform_sf_into_required_layout(qa[1], m_max, k, (1, 128, 128), g, True)
    sfb = dg.transform_sf_into_required_layout(qb[1], n, k, (1, 128, 128), g, False)
    masked_m = torch.tensor([5, 128, 64, 17], device='cuda', dtype=torch.int32)
    d = torch.zeros((g, m_max, n), device='cuda', dtype=torch.bfloat16)
    dg.m_grouped_fp8_gemm_nt_masked((qa[0], sfa), (qb[0], sfb), d, masked_m, 64)  # warm-up
    eager = d.clone()
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        d.zero_()
        with torch.cuda.graph(graph, stream=side):
            dg.m_grouped_fp8_gemm_nt_masked((qa[0], sfa), (qb[0], sfb), d, masked_m, 64)
    d.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(d, eager)
    # the graph reads masked_m at replay time
    masked_m.copy_(torch.tensor([128, 0, 1, 99], device='cuda', dtype=torch.int32))
    d.fill_(7.0)
    graph.replay()
    torch.cuda.synchronize()
    assert bool((d[1] == 7.0).all()) and float((d[0] != 7.0).float().mean()) > 0.99 and bool((d[2, 1:] == 7.0).all())


# ------------------------------------------------------------------------------------------------ full-size properties
def test_full_size_dense_properties(dg):
    """BASELINE configs[1] at full size (M=4096, N=4096, K=7168): the oracle is too slow here, so check exact algebraic
    properties of the kernel plus the reference's own tolerance against an FP32 GPU matmul of the dequantised operands."""
    m, n, k = 4096, 4096, 7168
    a, b, qa, qb = _quant_dense(m, n, k, seed=42)
    d = torch.empty((m, n), device='cuda', dtype=torch.float32)
    dg.fp8_gemm_nt(qa, qb, d)
    # (1) scales are powers of two: doubling token scales doubles every output exactly
    d2 = torch.empty_like(d)
    dg.fp8_gemm_nt((qa[0], qa[1] * 2), qb, d2)
    assert torch.equal(d2, d * 2)
    # (2) token rows are independent: permuting rows of A permutes rows of D, bit for bit
    perm = torch.randperm(m, device='cuda')
    d3 = torch.empty_like(d)
    dg.fp8_gemm_nt((qa[0][perm].contiguous(), qa[1][perm].contiguous()), qb, d3)
    assert torch.equal(d3, d[perm])
    # (3) zero tokens give exact zeros
    qa0 = qa[0].clone()
    qa0.view(torch.uint8)[100:200] = 0
    d4 = torch.empty_like(d)
    dg.fp8_gemm_nt((qa0, qa[1]), qb, d4)
    assert bool((d4[100:200] == 0).all()) and torch.equal(d4[200:], d[200:])
    # (4) FP32 matmul of the exactly dequantised operands (plain PyTorch reference for a floating-point kernel)
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = (qa[0].float() * qa[1].repeat_interleave(128, 1)) @ \
          (qb[0].float() * qb[1].repeat_interleave(128, 0).repeat_interleave(128, 1)).t()
    from deepgemm_b200.testing import calc_diff
    assert calc_diff(d, ref) < 1e-9
    assert ((d - ref).abs().max() / ref.abs().max()) < 1e-5
    assert calc_diff(d, a.float() @ b.float().t()) < 1e-3          # reference test tolerance (unquantised inputs)


def test_golden_outputs_of_the_reference_kernel(dg):
    """tests/golden/gpu_golden.*.pt hold outputs of the reference's own SM100 kernel (generated on a B200 by
    tests/golden/make_golden_gpu.py). Same FP8 inputs + scale factors -> the outputs must match bit for bit."""
    from golden import store
    golden = store.load(os.path.join(HERE, 'golden'), 'gpu_golden')
    for case in golden['dense']:
        qa = (case['a'].cuda().view(torch.float8_e4m3fn), case['sfa'].cuda())
        qb = (case['b'].cuda().view(torch.float8_e4m3fn), case['sfb'].cuda())
        d = torch.empty(case['d'].shape, device='cuda', dtype=case['d'].dtype)
        c = case.get('c')
        os.environ['DGB200_SPLITS'] = '1'   # bitwise comparison: same K order as the reference (no split-K)
        try:
            if c is not None:
                d.copy_(c.cuda())
                dg.fp8_gemm_nt(qa, qb, d, c=d)
            else:
                dg.fp8_gemm_nt(qa, qb, d)
        finally:
            os.environ.pop('DGB200_SPLITS', None)
        assert torch.equal(d.cpu(), case['d']), case['name']
    for case in golden.get('dense_tn', []):
        a_t = (case['a_t'].cuda().view(torch.float8_e4m3fn), case['sfa_t'].cuda())
        b_t = (case['b_t'].cuda().view(torch.float8_e4m3fn), case['sfb_t'].cuda())
        d = torch.empty(case['d'].shape, device='cuda', dtype=case['d'].dtype)
        dg.fp8_gemm_tn(a_t, b_t, d)
        assert torch.equal(d.cpu(), case['d']), case['name']
    for case in golden.get('k_grouped', []):
        a = (case['a'].cuda().view(torch.float8_e4m3fn), case['sfa'].cuda())
        b = (case['b'].cuda().view(torch.float8_e4m3fn), case['sfb'].cuda())
        d = case['c'].cuda().clone()
        dg.set_mk_alignment_for_contiguous_layout(case['k_alignment'])
        try:
            dg.k_grouped_fp8_gemm_tn_contiguous(a, b, d, case['ks'], torch.tensor(case['ks'], device='cuda', dtype=torch.int32),
                                                c=d, recipe=(1, 1, case['gran_k']))
        finally:
            dg.set_mk_alignment_for_contiguous_layout(128)
        assert torch.equal(d.cpu(), case['d']), case['name']
    for case in golden.get('masked', []):
        qa = (case['a'].cuda().view(torch.float8_e4m3fn), case['sfa'].cuda())
        qb = (case['b'].cuda().view(torch.float8_e4m3fn), case['sfb'].cuda())
        mm = case['masked_m'].cuda()
        d = torch.zeros(case['d'].shape, device='cuda', dtype=torch.bfloat16)
        dg.m_grouped_fp8_gemm_nt_masked(qa, qb, d, mm, case['expected_m'])
        for gi, mg in enumerate(case['masked_m'].tolist()):
            assert torch.equal(d[gi, :mg].cpu(), case['d'][gi, :mg]), case['name']
    for case in golden.get('contiguous', []):
        qa = (case['a'].cuda().view(torch.float8_e4m3fn), case['sfa'].cuda())
        qb = (case['b'].cuda().view(torch.float8_e4m3fn), case['sfb'].cuda())
        d = torch.zeros(case['d'].shape, device='cuda', dtype=torch.bfloat16)
        dg.set_mk_alignment_for_contiguous_layout(case['alignment'])
        try:
            dg.m_grouped_fp8_gemm_nt_contiguous(qa, qb, d, case['layout'].cuda(), use_psum_layout=case['psum'])
        finally:
            dg.set_mk_alignment_for_contiguous_layout(128)
        valid = case['valid']
        assert torch.equal(d.cpu()[valid], case['d'][valid]), case['name']
