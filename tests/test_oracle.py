"""CPU: pin the oracle (oracle/blockwise.py) and the caller-side helpers (deepgemm_b200.utils) against golden vectors
produced by the REFERENCE'S OWN python code (tests/golden/make_golden_cpu.py). Bit-exact for bytes / integers."""
import torch

from deepgemm_b200.testing import calc_diff
from deepgemm_b200.utils import math as umath
from oracle import blockwise as oracle


def test_ceil_to_ue8m0_matches_reference(cpu_golden):
    g = cpu_golden['ue8m0']
    assert torch.equal(umath.ceil_to_ue8m0(g['x']).view(torch.int32), g['y'].view(torch.int32))


def test_quantizers_match_reference_bitwise(cpu_golden):
    for case in cpu_golden['quant']:
        x, use, gk = case['x'], case['use_ue8m0'], case['gran_k']
        if case['kind'] == 'token':
            q, sf = umath.per_token_cast_to_fp8(x, use, gk)
        elif case['kind'] == 'token_packed':
            q, sf = umath.per_token_cast_to_fp8(x, use, gk, use_packed_ue8m0=True)
        elif case['kind'] == 'block':
            q, sf = umath.per_block_cast_to_fp8(x, use, gk)
        else:
            q, sf = umath.per_channel_cast_to_fp8(x, use, gk)
        assert torch.equal(q.view(torch.uint8), case['q']), case['kind']
        assert sf.dtype == case['sf'].dtype and sf.shape == case['sf'].shape
        assert torch.equal(sf.contiguous().view(torch.int32), case['sf'].contiguous().view(torch.int32)), case['kind']


def test_packed_sf_wire_format_matches_reference(cpu_golden):
    for case in cpu_golden['pack']:
        packed = oracle.pack_sf_ue8m0_mn_major(case['sf'])
        assert tuple(packed.shape) == case['shape']
        assert tuple(packed.stride()) == case['stride']
        assert torch.equal(packed, case['packed'])
        # and back
        sf_k = case['sf'].shape[-1]
        assert torch.equal(oracle.unpack_sf_ue8m0(packed, sf_k).view(torch.int32), case['sf'].view(torch.int32))


def test_pack_ue8m0_to_int_is_the_k_major_view_of_the_wire_format(cpu_golden):
    for case in cpu_golden['pack']:
        sf = case['sf']
        if sf.shape[-1] % 4:
            continue
        assert torch.equal(umath.pack_ue8m0_to_int(sf), case['dense'])


def test_calc_diff_matches_reference(cpu_golden):
    for case in cpu_golden['calc_diff']:
        assert abs(calc_diff(case['x'], case['y']) - case['d']) < 1e-12


def _inputs(m, n, k, seed=0):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn((m, k), generator=g).to(torch.bfloat16)
    b = torch.randn((n, k), generator=g).to(torch.bfloat16)
    return a, b, umath.per_token_cast_to_fp8(a, True), umath.per_block_cast_to_fp8(b, True)


def test_config1_plumbing_128cube():
    """BASELINE config 1: fp8_gemm_nt M=N=K=128 against the torch-CPU BF16-emulated blockwise GEMM, and against the
    FP32 matmul of the unquantised inputs with the reference's own tolerance (tests/test_fp8_fp4.py:53-55)."""
    a, b, qa, qb = _inputs(128, 128, 128)
    d = oracle.fp8_gemm_nt(qa, qb)
    emu = oracle.bf16_emulated_gemm_nt(qa, qb)
    assert calc_diff(d, emu) < 1e-5
    assert calc_diff(d, a.float() @ b.float().t()) < 1e-3


def test_oracle_accepts_packed_and_fp32_sfs_identically():
    a, b, qa, qb = _inputs(96, 256, 384, seed=1)
    d0 = oracle.fp8_gemm_nt(qa, qb)
    sfa = oracle.pack_sf_ue8m0_mn_major(qa[1])
    sfb = oracle.pack_sf_ue8m0_mn_major(qb[1].repeat_interleave(128, 0)[:256])
    d1 = oracle.fp8_gemm_nt((qa[0], sfa), (qb[0], sfb), recipe=(1, 1, 128))
    assert torch.equal(d0, d1)


def test_oracle_linearity_in_scale_factors():
    """Doubling every token scale doubles the (FP32) result exactly: scales are powers of two."""
    a, b, qa, qb = _inputs(32, 128, 256, seed=2)
    d0 = oracle.fp8_gemm_nt(qa, qb, out_dtype=torch.float32)
    d1 = oracle.fp8_gemm_nt((qa[0], qa[1] * 2), qb, out_dtype=torch.float32)
    assert torch.equal(d1, d0 * 2)


def test_oracle_accumulate_and_empty_semantics():
    a, b, qa, qb = _inputs(16, 128, 128, seed=3)
    c32 = torch.randn(16, 128)
    d = oracle.fp8_gemm_nt(qa, qb, out_dtype=torch.float32, c=c32)
    assert torch.equal(d, oracle.fp8_gemm_nt(qa, qb, out_dtype=torch.float32) + c32)
    cb = c32.to(torch.bfloat16)
    db = oracle.fp8_gemm_nt(qa, qb, c=cb)
    assert torch.equal(db, (oracle.fp8_gemm_nt(qa, qb).float() + cb.float()).to(torch.bfloat16))
    # K == 0 -> D = C or 0 (csrc/apis/gemm.hpp:36-40)
    e = (torch.empty((4, 0), dtype=torch.float8_e4m3fn), torch.empty((4, 0)))
    f = (torch.empty((8, 0), dtype=torch.float8_e4m3fn), torch.empty((1, 0)))
    assert torch.equal(oracle.fp8_gemm_nt(e, f), torch.zeros((4, 8), dtype=torch.bfloat16))


def test_grouped_oracles_agree_with_per_group_dense():
    g, n, k = 3, 128, 256
    gen = torch.Generator().manual_seed(4)
    ms = [40, 0, 100]
    align_m = 64
    rows, layout = [], []
    for gi, mg in enumerate(ms):
        am = oracle.align(mg, align_m)
        x = torch.randn((am, k), generator=gen).to(torch.bfloat16)
        x[mg:] = 0
        rows.append(x)
        layout += [gi] * mg + [-1] * (am - mg)
    a = torch.cat(rows)
    b = torch.randn((g, n, k), generator=gen).to(torch.bfloat16)
    qa = umath.per_token_cast_to_fp8(a, True)
    qb_list = [umath.per_block_cast_to_fp8(b[i], True) for i in range(g)]
    qb = (torch.stack([q[0] for q in qb_list]), torch.stack([q[1] for q in qb_list]))
    d, valid = oracle.m_grouped_fp8_gemm_nt_contiguous(qa, qb, torch.tensor(layout, dtype=torch.int32))
    start = 0
    for gi, mg in enumerate(ms):
        want = oracle.fp8_gemm_nt((qa[0][start:start + mg], qa[1][start:start + mg]), qb_list[gi])
        assert torch.equal(d[start:start + mg], want)
        assert bool(valid[start:start + mg].all())
        start += oracle.align(mg, align_m)
    # psum layout describes the same problem
    ends, s = [], 0
    for mg in ms:
        ends.append(s + mg)
        s = oracle.align(s + mg, align_m)
    d2, valid2 = oracle.m_grouped_fp8_gemm_nt_contiguous(qa, qb, torch.tensor(ends, dtype=torch.int32),
                                                        use_psum_layout=True, alignment=align_m)
    assert torch.equal(valid, valid2) and torch.equal(d[valid], d2[valid2])
    # masked layout
    a3 = torch.randn((g, 64, k), generator=gen).to(torch.bfloat16)
    q3 = [umath.per_token_cast_to_fp8(a3[i], True) for i in range(g)]
    qa3 = (torch.stack([q[0] for q in q3]), torch.stack([q[1] for q in q3]))
    mm = torch.tensor([10, 0, 64], dtype=torch.int32)
    dm = oracle.m_grouped_fp8_gemm_nt_masked(qa3, qb, mm)
    for gi, mg in enumerate(mm.tolist()):
        want = oracle.fp8_gemm_nt((q3[gi][0][:mg], q3[gi][1][:mg]), qb_list[gi])
        assert torch.equal(dm[gi, :mg], want)


# ------------------------------------------------------------------------------------------------ oracle vs the reference KERNEL
def _gpu_golden():
    import os
    from golden import store
    return store.load(os.path.join(os.path.dirname(__file__), 'golden'), 'gpu_golden')


def _assert_oracle_close(got, ref_out, what):
    """Oracle (FP64 accumulation) versus the reference's SM100 kernel output (FP32 accumulation in tensor-core order): the
    stated tolerance of DESIGN.md section 2 -- FP32 outputs within 1e-5 * max|D|, BF16 outputs within one BF16 rounding
    step of the value plus that noise, on at most 2 % of the elements."""
    assert got.shape == ref_out.shape and got.dtype == ref_out.dtype, what
    assert calc_diff(got, ref_out) < 1e-6, what
    if got.dtype == torch.float32:
        assert ((got - ref_out).abs().max() / ref_out.abs().max().clamp(min=1.0)) < 1e-5, what
    else:
        mism = got != ref_out
        assert mism.float().mean() <= 0.02, what
        err = (got.float() - ref_out.float()).abs()
        mag = ref_out.float().abs()
        assert bool((err <= mag * 2.0 ** -7 + 1e-5 * mag.max()).all()), what


def test_oracle_reproduces_the_reference_kernels_golden_outputs():
    """Direct pin of the CPU restatement on the outputs of the UNMODIFIED reference kernel (tests/golden/gpu_golden.*.pt,
    made on a B200 by tests/golden/make_golden_gpu.py): dense (+ C accumulation, BF16 and FP32), masked, contiguous
    (+ psum), MN-major (tn) and the K-grouped weight gradient."""
    g = _gpu_golden()
    f8 = lambda t: t.view(torch.float8_e4m3fn)  # noqa: E731
    for case in g['dense']:
        c = case.get('c')
        got = oracle.fp8_gemm_nt((f8(case['a']), case['sfa']), (f8(case['b']), case['sfb']), out_dtype=case['d'].dtype, c=c)
        if c is not None and case['d'].dtype == torch.bfloat16:
            continue   # BF16 accumulate: checked below with the magnitude of product + C (cancellation)
        _assert_oracle_close(got, case['d'], case['name'])
    for case in g['dense']:
        c = case.get('c')
        if c is None or case['d'].dtype != torch.bfloat16:
            continue
        got = oracle.fp8_gemm_nt((f8(case['a']), case['sfa']), (f8(case['b']), case['sfb']), out_dtype=torch.bfloat16, c=c)
        prod = oracle.fp8_gemm_nt((f8(case['a']), case['sfa']), (f8(case['b']), case['sfb']), out_dtype=torch.float32)
        err = (got.float() - case['d'].float()).abs()
        mag = prod.abs() + c.float().abs()
        assert bool((err <= mag * 2.0 ** -7 + 1e-5 * mag.max()).all()), case['name']
    for case in g.get('dense_tn', []):
        a = (f8(case['a_t']).t(), case['sfa_t'].t())
        b = (f8(case['b_t']).t(), case['sfb_t'].t())
        got = oracle.fp8_gemm_nt((a[0].contiguous(), a[1].contiguous()), (b[0].contiguous(), b[1].contiguous()), out_dtype=case['d'].dtype)
        _assert_oracle_close(got, case['d'], case['name'])
    for case in g.get('masked', []):
        got = oracle.m_grouped_fp8_gemm_nt_masked((f8(case['a']), case['sfa']), (f8(case['b']), case['sfb']), case['masked_m'])
        for gi, mg in enumerate(case['masked_m'].tolist()):
            if mg:
                _assert_oracle_close(got[gi, :mg], case['d'][gi, :mg], case['name'])
    for case in g.get('contiguous', []):
        got, valid = oracle.m_grouped_fp8_gemm_nt_contiguous((f8(case['a']), case['sfa']), (f8(case['b']), case['sfb']), case['layout'],
                                                             use_psum_layout=case['psum'], alignment=case['alignment'])
        assert torch.equal(valid, case['valid'])
        _assert_oracle_close(got[valid], case['d'][valid], case['name'])
    for case in g.get('k_grouped', []):
        got = oracle.k_grouped_fp8_gemm_tn_contiguous((f8(case['a']), case['sfa']), (f8(case['b']), case['sfb']), case['c'], case['ks'],
                                                      gran_k=case['gran_k'])
        _assert_oracle_close(got, case['d'], case['name'])


def test_golden_fixture_files_stay_within_1_mb():
    import os
    from golden import store
    golden = os.path.join(os.path.dirname(__file__), 'golden')
    sizes = {f: os.path.getsize(os.path.join(golden, f)) for f in os.listdir(golden) if os.path.isfile(os.path.join(golden, f))}
    assert max(sizes.values()) <= store.PART_LIMIT, sizes
