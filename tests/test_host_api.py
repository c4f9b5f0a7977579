"""CPU: the C-ABI library loads and exports every symbol include/dgb200.h declares; host-side logic (knobs,
heuristics, argument validation, error behaviour) works without a GPU. No compute calls here."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    from deepgemm_b200 import _lib
    _lib.build()
    return _lib


def _declared_symbols():
    text = open(os.path.join(REPO, 'include', 'dgb200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(dgb200_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol(lib):
    handle = ctypes.CDLL(lib.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(handle, name), f'{name} declared in include/dgb200.h but not exported'
    assert sorted(lib.SIGNATURES) == declared, 'python binding table and header disagree'


def test_version_and_knobs_roundtrip(lib):
    import deepgemm_b200 as dg
    assert lib.lib().dgb200_version() == 100
    dg.set_tc_util(80)
    assert dg.get_tc_util() == 80
    dg.set_tc_util(100)
    dg.set_pdl(True)
    assert dg.get_pdl() is True
    dg.set_pdl(False)
    assert dg.get_mk_alignment_for_contiguous_layout() == 128  # legacy default, heuristics/runtime.hpp:10
    dg.set_mk_alignment_for_contiguous_layout(224)
    assert dg.get_mk_alignment_for_contiguous_layout() == 224
    dg.set_mk_alignment_for_contiguous_layout(128)
    # any 0 <= n <= SM count like the reference (jit/device_runtime.hpp:103-105); 0 = all SMs; an odd budget is
    # accepted (the reference only trips over it later, heuristics/config.hpp:47) and rounded down to whole CTA pairs
    dg.set_num_sms(147)
    assert lib.lib().dgb200_get_num_sms() == 147
    dg.set_num_sms(0)
    # 0 reads back as 0 until the library has set up a device (the GPU tests before this one do in a whole-suite run),
    # from then on as that device's SM count
    n = lib.lib().dgb200_get_num_sms()
    assert n == 0 or n == torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    with pytest.raises(RuntimeError):
        dg.set_num_sms(-2)
    with pytest.raises(RuntimeError):
        dg.set_mk_alignment_for_contiguous_layout(100)


def test_alignment_helpers_match_reference_formulas(lib):
    import deepgemm_b200 as dg
    # csrc/utils/math.hpp:23-27
    assert [dg.get_tma_aligned_size(x, 4) for x in (1, 4, 5, 4097)] == [4, 4, 8, 4100]
    assert dg.get_tma_aligned_size(17, 1) == 32
    # heuristics/runtime.hpp:47-57 (arch 10)
    assert dg.get_theoretical_mk_alignment_for_contiguous_layout() == 224
    assert dg.get_theoretical_mk_alignment_for_contiguous_layout(1000) == 224
    assert dg.get_theoretical_mk_alignment_for_contiguous_layout(100) == 128
    assert dg.get_theoretical_mk_alignment_for_contiguous_layout(20) == 32


def test_heuristics_baseline_shapes(lib):
    """Plan for the BASELINE.json shapes: valid tile heights, pipelines that fit 227 KB, CTA pairs."""
    for m in (1, 64, 128, 512, 4096):
        cfg = lib.plan(0, m, 4096, 7168)
        assert cfg['block_m'] % 16 == 0 and 16 <= cfg['block_m'] <= 240
        cs = cfg['cluster_split']
        assert cfg['cluster'] == (cs or 2) and cfg['num_sms'] == 148 and cs in (0, 2, 4)
        assert cfg['smem_bytes'] <= 232448 and cfg['num_stages'] >= 4
        if cs:      # cluster split-K: few output tiles, K cut over the CTAs of a cluster, token chunks of 16 columns per CTA
            assert m <= 256 and cfg['num_splits'] == cs and cfg['block_m'] % (16 * cs) == 0 and cfg['num_tiles'] <= 148
        else:
            assert cfg['block_m'] - 16 < max(m, 16)
    assert lib.plan(0, 64, 4096, 7168)['cluster_split'] == 4       # the decode-sized headline shapes stream K from all SMs
    assert lib.plan(0, 512, 4096, 7168)['cluster_split'] == 0 and lib.plan(0, 4096, 4096, 7168)['cluster_split'] == 0
    big = lib.plan(0, 4096, 4096, 7168)
    assert big['block_m'] >= 192                      # compute-bound shape wants tall tiles
    cont = lib.plan(1, 32768, 4096, 7168, 256, 128, 128)
    assert 128 % cont['block_m'] == 0                 # a tile never straddles two experts
    masked = lib.plan(2, 128, 7168, 2048, 256, 64)
    assert masked['block_m'] <= 128


def test_python_api_validation_errors_without_gpu(lib):
    """Contract violations raise RuntimeError before anything touches CUDA (DG_HOST_ASSERT -> RuntimeError)."""
    import deepgemm_b200 as dg
    a = torch.zeros((8, 128), dtype=torch.float8_e4m3fn)
    b = torch.zeros((16, 128), dtype=torch.float8_e4m3fn)
    sfa, sfb = torch.ones((8, 1)), torch.ones((1, 1))
    with pytest.raises(RuntimeError, match='m == m_'):
        dg.fp8_gemm_nt((a, sfa), (b, sfb), torch.zeros((8, 32), dtype=torch.bfloat16))
    with pytest.raises(RuntimeError, match='bfloat16 or float'):
        dg.fp8_gemm_nt((a, sfa), (b, sfb), torch.zeros((8, 16), dtype=torch.float16))
    with pytest.raises(RuntimeError, match='FP4'):
        dg.fp8_gemm_nt((a.view(torch.int8), sfa), (b, sfb), torch.zeros((8, 16), dtype=torch.bfloat16))
    with pytest.raises(RuntimeError, match='row-major'):
        dg.fp8_gemm_nt((a, sfa), (b, sfb), torch.zeros((16, 8), dtype=torch.bfloat16).t())
    # empty problems return before any device work (gemm.hpp:22-23)
    dg.fp8_gemm_nt((a[:0], sfa[:0]), (b, sfb), torch.zeros((0, 16), dtype=torch.bfloat16))
    # k == 0 -> D = C (gemm.hpp:36-40)
    d = torch.ones((8, 16), dtype=torch.bfloat16)
    c = torch.full((8, 16), 3.0, dtype=torch.bfloat16)
    dg.fp8_gemm_nt((a[:, :0], sfa[:, :0]), (b[:, :0], sfb[:, :0]), d, c=c)
    assert torch.equal(d, c)
    with pytest.raises(RuntimeError, match='grouped_layout'):
        dg.m_grouped_fp8_gemm_nt_contiguous((a, sfa), (b.view(1, 16, 128), sfb.view(1, 1, 1)),
                                            torch.zeros((8, 16), dtype=torch.bfloat16),
                                            torch.zeros(3, dtype=torch.int32))
    with pytest.raises(RuntimeError, match='Unsupported architecture'):
        dg.k_grouped_fp8_gemm_nt_contiguous(None, None, None, None, None)


def test_aliases_and_dropin_module(lib):
    import deep_gemm
    import deepgemm_b200 as dg
    assert deep_gemm.fp8_gemm_nt is dg.fp8_gemm_nt
    assert deep_gemm.fp8_fp4_gemm_nt is dg.fp8_gemm_nt
    assert deep_gemm.fp8_m_grouped_gemm_nt_masked is dg.m_grouped_fp8_gemm_nt_masked
    from deep_gemm.utils import per_token_cast_to_fp8  # noqa: F401
    from deep_gemm.testing import calc_diff  # noqa: F401
    for name in ('fp8_gemm_nt', 'fp8_gemm_nn', 'fp8_gemm_tn', 'fp8_gemm_tt', 'm_grouped_fp8_gemm_nt_contiguous',
                 'm_grouped_fp8_gemm_nn_contiguous', 'm_grouped_fp8_gemm_nt_masked', 'k_grouped_fp8_gemm_tn_contiguous',
                 'transform_sf_into_required_layout', 'get_mn_major_tma_aligned_packed_ue8m0_tensor', 'set_num_sms',
                 'get_num_sms', 'set_tc_util', 'set_pdl', 'get_mk_alignment_for_contiguous_layout'):
        assert hasattr(deep_gemm, name), name


def test_import_does_not_touch_cuda():
    """The reference guarantees import-then-fork safety (tests/test_lazy_init.py); so do we."""
    code = ('import torch, deepgemm_b200, deep_gemm; from deepgemm_b200 import _lib; _lib.lib(); '
            'assert not torch.cuda.is_initialized(); print("ok")')
    out = subprocess.run([sys.executable, '-c', code], cwd=REPO, capture_output=True, text=True)
    assert out.returncode == 0 and 'ok' in out.stdout, out.stderr


def test_product_path_never_imports_the_oracle():
    for root, _, files in os.walk(os.path.join(REPO, 'deepgemm_b200')):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                text = open(os.path.join(root, f)).read()
                assert 'import oracle' not in text and 'from oracle' not in text, f


def test_gemm_kernels_keep_tma_operands_in_uniform_registers():
    """Build sanity (no GPU): the TMA producer / MMA issuer run as one elected thread; if ptxas loses that fact it wraps
    every UTMALDG in an R2UR.BROADCAST 'waterfall' loop, which measured ~2x slower per k-block on B200. None allowed."""
    import shutil
    import subprocess
    from deepgemm_b200 import _lib
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    sass = subprocess.run([cuobjdump, '-sass', _lib.build()], capture_output=True, text=True, check=True).stdout
    kernels = sass.split('Function : ')[1:]
    gemm = [k for k in kernels if 'fp8_gemm_kernel' in k.split('\n', 1)[0]]
    assert len(gemm) >= 40
    bad = [k.split('\n', 1)[0] for k in gemm if 'R2UR.BROADCAST' in k]
    assert not bad, bad[:3]
    assert all('UTMALDG' in k and ('UTCQMMA' in k or 'UTCOMMA' in k or 'UTCHMMA' in k or 'UTCMMA' in k or 'UTC' in k) for k in gemm)


def test_ep_buffer_layout_and_argument_checks(lib):
    """Host side of the expert-parallel entry points (no GPU): the layout is a pure function, regions are ordered,
    aligned and large enough; bad arguments are rejected with the library's error text."""
    import ctypes
    L = lib.lib()
    world, g, cap, k = 4, 256, 10240, 7168
    total = L.dgb200_ep_buffer_bytes(world, g, cap, k)
    offs = (ctypes.c_int64 * 6)()
    assert L.dgb200_ep_buffer_offsets(world, g, cap, k, offs) == 0
    a, sfa, psum, counts, rows, overflow = list(offs)
    assert 0 < rows < overflow < 256 < psum and psum % 1024 == 0 and counts % 1024 == 0
    assert sfa % 1024 == 0 and a % 1024 == 0 and sfa + 4 * ((k + 511) // 512) * cap <= a and a + cap * k <= total
    assert total < a + cap * k + 4096
    assert L.dgb200_ep_buffer_bytes(0, g, cap, k) == 0
    bufs = (ctypes.c_void_p * world)(*([4096] * world))
    # experts must divide over the ranks; K must be a multiple of 16; ids are int32 or int64
    for bad in (dict(g=255), dict(k=7170), dict(idb=2)):
        rc = L.dgb200_ep_dispatch(4096, k, 4096, 14, 1, 4096, bad.get('idb', 8), 16, 1, bad.get('k', k), bad.get('g', g), 0, world,
                                  bufs, cap, 128, 4096, 4096, 1, None)
        assert rc != 0 and b'Assertion error' in L.dgb200_last_error()


def test_dense_plan_balances_rounds_of_cta_pairs(lib):
    """M = N = 4096 on 74 CTA pairs: uniform 240-row tiles would leave a 16-row m-block behind (17 x 240 + 16); the planner
    makes 18 m-blocks of 240 / 224 rows (288 tiles, 3.89 rounds). It weighs rows by tile height (taller tiles move fewer
    operand bytes per FLOP, which is clock under the power cap): 23 m-blocks of 192 / 176 rows fill 4.97 rounds more evenly
    but measured 1 % slower. M = 6144 keeps shorter tiles: 32 m-blocks of 192 rows are 6.92 rounds."""
    cfg = lib.plan(0, 4096, 4096, 7168)
    assert cfg['block_m'] == 240 and cfg['cluster'] == 2 and cfg['num_splits'] == 1
    assert cfg['num_tiles'] == 18 * 16                  # 4 x 240 + 14 x 224 rows = 4096, times 16 column pairs
    assert lib.plan(0, 8192, 4096, 7168)['block_m'] == 224          # 37 m-blocks of 224 / 208 rows: 8 rounds
    small = lib.plan(0, 512, 4096, 7168)
    assert small['block_m'] == 128                       # below 1024 rows the tile height is chosen by the cost model alone


def test_plan_picks_pair_split_k_and_the_staged_epilogue_where_measured(lib):
    """Round-2 heuristics (DESIGN.md section 4 / 10): medium M runs as two CTA-pair K slices while all clusters of 4 fit one
    wave; tall tiles with a long K loop take the TMA-store epilogue unless it would cost a pipeline stage."""
    c = lib.plan(0, 192, 4096, 7168)
    assert (c['cluster'], c['cluster_split'], c['block_m']) == (4, 2, 96)
    c = lib.plan(0, 256, 4096, 7168)
    assert (c['cluster'], c['cluster_split'], c['block_m']) == (4, 2, 128)
    c = lib.plan(0, 256, 2112, 7168)
    assert (c['cluster'], c['cluster_split'], c['block_m']) == (4, 2, 96)      # 27 clusters; 64-row tiles would need 36 > 32
    c = lib.plan(0, 320, 4096, 7168)
    assert c['cluster_split'] == 0 and c['cluster'] == 2                         # 48 clusters: no longer one wave
    c = lib.plan(0, 256, 7168, 2048)
    assert c['cluster_split'] == 0                                               # short K: the exchange does not pay
    c = lib.plan(0, 64, 4096, 7168)
    assert (c['cluster'], c['cluster_split']) == (4, 4)                          # small M: four single-CTA slices
    big = lib.plan(0, 4096, 7168, 2048)
    assert big['tma_store'] == 1 and big['block_m'] >= 176 and big['num_stages'] >= 6
    assert lib.plan(0, 4096, 32768, 512)['tma_store'] == 0                       # epilogue-bound: direct stores
    assert lib.plan(0, 512, 4096, 7168)['tma_store'] == 0                        # 128-row tiles: the staging would cost a stage
    assert lib.plan(1, 32768, 4096, 7168, 256, 128, 128)['tma_store'] == 0       # contiguous, 128-row tiles
    assert all(lib.plan(0, m, 4096, 7168)['swap_ab'] == 0 for m in (1, 64, 512, 4096))   # second orientation: not for these
    sw = lib.plan(0, 512, 7168, 2048)      # 28 x 5 tiles = two rounds of pairs; 2 x 32 tiles of 256 tokens x 224 weights = one
    assert (sw['swap_ab'], sw['block_m'], sw['cluster'], sw['tma_store'], sw['num_tiles']) == (1, 224, 2, 1, 64)
    assert lib.plan(0, 256, 7168, 2048)['swap_ab'] == 0 and lib.plan(0, 1024, 7168, 2048)['swap_ab'] == 0


def test_prepacked_scale_factor_pair_memo_notices_a_changed_layout():
    """The per-call fast path remembers the last validated pair of pre-packed scale-factor tensors by identity; shapes and
    strides are still compared on every call, so an in-place transpose (or any other tensor) goes through the full checks."""
    import torch
    from deepgemm_b200 import layout
    m, n, k = 64, 256, 1024
    sfa = torch.zeros((k // 512, m), dtype=torch.int32).t()
    sfb = torch.zeros((k // 512, n), dtype=torch.int32).t()
    first = layout.transform_sf_pair_into_required_layout(sfa, sfb, m, n, k, None, None, None, None, None)
    again = layout.transform_sf_pair_into_required_layout(sfa, sfb, m, n, k, None, None, None, None, None)
    assert again == first and again[0] is sfa and again[1] is sfb and first[2:] == (128, 128)
    import gc
    import weakref
    probe = torch.zeros((k // 512, m), dtype=torch.int32).t()
    layout.transform_sf_pair_into_required_layout(probe, sfb, m, n, k, None, None, None, None, None)
    alive = weakref.ref(probe)
    del probe
    gc.collect()
    assert alive() is None, 'the memo keeps a validated tensor alive' 
    with pytest.raises(RuntimeError):
        layout.transform_sf_pair_into_required_layout(sfa, sfb, m + 4, n, k, None, None, None, None, None)     # other problem size
    other = torch.zeros((m, k // 512), dtype=torch.int32)                                                         # K-major storage: not TMA-ready
    with pytest.raises(RuntimeError):
        layout.transform_sf_pair_into_required_layout(other, sfb, m, n, k, None, None, None, None, None)
    assert layout.transform_sf_pair_into_required_layout(sfa, sfb, m, n, k, None, None, None, None, None)[0] is sfa
    sfa.t_()                                                                                                       # same object, new layout
    with pytest.raises(RuntimeError):
        layout.transform_sf_pair_into_required_layout(sfa, sfb, m, n, k, None, None, None, None, None)


def test_tools_and_bench_compile():
    """bench.py, __graft_entry__.py and every helper under tools/ at least parse (they only run on the GPU box)."""
    import glob
    files = [os.path.join(REPO, 'bench.py'), os.path.join(REPO, '__graft_entry__.py')] + sorted(glob.glob(os.path.join(REPO, 'tools', '*.py')))
    assert len(files) > 10
    for f in files:
        compile(open(f).read(), f, 'exec')


def test_bench_dump_outputs_stays_within_64_mb_and_samples_the_same_rows(tmp_path):
    """bench.py --dump-outputs: float32 files, 64 MB in all at the benchmark's shapes; the small outputs are whole, the
    largest keeps a sorted, seeded sample of as many rows as the rest of the budget holds, so two runs write identical files."""
    import numpy as np

    import bench
    probs = [dict(m=m, n=n, k=k, d=torch.randn((m, n), generator=torch.Generator().manual_seed(m)).to(torch.bfloat16))
             for m, n, k in bench.DENSE_SHAPES]
    for run in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / run), probs)
    total = sum(f.stat().st_size for f in (tmp_path / 'a').iterdir())
    assert 60_000_000 < total <= 64_000_000
    sampled = 0
    for p in probs:
        name = f"d_{p['m']}x{p['n']}x{p['k']}.npy"
        got = np.load(tmp_path / 'a' / name)
        assert got.dtype == np.float32 and got.shape[1] == p['n']
        assert np.array_equal(got, np.load(tmp_path / 'b' / name))
        full = p['d'].float().numpy()
        if got.shape[0] == p['m']:
            assert np.array_equal(got, full)
            continue
        sampled += 1
        row_of = {full[i].tobytes(): i for i in range(p['m'])}
        picked = [row_of[r.tobytes()] for r in got]
        assert picked == sorted(set(picked))
    assert sampled == 1
