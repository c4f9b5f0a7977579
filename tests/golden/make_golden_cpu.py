"""Generate CPU golden vectors FROM THE REFERENCE'S OWN PYTHON CODE (run in the build container, where
/root/reference exists; the outputs are committed, the GPU box never needs the reference for them).

Sources executed (unmodified, imported from the reference install oracle/_ref which oracle/build_ref.sh creates):
  * deep_gemm/utils/math.py:13-61    ceil_to_ue8m0, pack_ue8m0_to_int, per_token/per_block/per_channel casts
  * deep_gemm/testing/numeric.py:5-11 calc_diff
  * tests/test_layout.py:20-42        get_mn_major_tma_aligned_packed_ue8m0_tensor_torch_impl -- the reference's own
                                      bit-exact statement of the packed-UE8M0 wire format (loaded by path)
Output: tests/golden/cpu_golden.*.pt (tests/golden/store.py)
"""
import importlib.util
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF_INSTALL = os.path.join(REPO, 'oracle', '_ref')
REF_SRC = os.environ.get('REF_SRC', '/root/reference')


def load_reference():
    sys.path.insert(0, REF_INSTALL)
    sys.path.insert(0, os.path.join(REF_SRC, 'tests'))  # for `generators`, imported by test_layout.py
    import deep_gemm  # the reference package (imports fine without a GPU)
    assert REF_INSTALL in deep_gemm.__file__
    spec = importlib.util.spec_from_file_location('ref_test_layout', os.path.join(REF_SRC, 'tests', 'test_layout.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return deep_gemm, mod


def main():
    ref, ref_layout = load_reference()
    from deep_gemm.utils import math as rmath
    from deep_gemm.testing.numeric import calc_diff
    out = {'quant': [], 'pack': [], 'calc_diff': [], 'ue8m0': None}

    torch.manual_seed(20260921)
    x = torch.cat([torch.randn(4096), torch.tensor([0.0, 1e-30, 1.0, 2.0, 3.0, 448.0, 1e30, 2.0 ** -126, 2.0 ** 127])])
    out['ue8m0'] = {'x': x, 'y': rmath.ceil_to_ue8m0(x)}

    for (m, k, gran_k) in [(7, 128, 128), (64, 384, 128), (33, 200, 128), (16, 96, 32)]:
        xin = (torch.randn(m, k) * torch.rand(m, 1) * 8).to(torch.bfloat16)
        for use_ue8m0 in (False, True):
            q, sf = rmath.per_token_cast_to_fp8(xin, use_ue8m0=use_ue8m0, gran_k=gran_k)
            out['quant'].append({'kind': 'token', 'x': xin, 'use_ue8m0': use_ue8m0, 'gran_k': gran_k,
                                 'q': q.view(torch.uint8), 'sf': sf})
        q, sf = rmath.per_token_cast_to_fp8(xin, use_ue8m0=True, gran_k=gran_k, use_packed_ue8m0=(sf.size(-1) % 4 == 0))
        if sf.dtype == torch.int32:
            out['quant'].append({'kind': 'token_packed', 'x': xin, 'use_ue8m0': True, 'gran_k': gran_k,
                                 'q': q.view(torch.uint8), 'sf': sf})
    for (m, k) in [(128, 128), (200, 300), (256, 512)]:
        xin = (torch.randn(m, k) * 3).to(torch.bfloat16)
        for use_ue8m0 in (False, True):
            q, sf = rmath.per_block_cast_to_fp8(xin, use_ue8m0=use_ue8m0)
            out['quant'].append({'kind': 'block', 'x': xin, 'use_ue8m0': use_ue8m0, 'gran_k': 128,
                                 'q': q.view(torch.uint8), 'sf': sf})
    for (k, n, gran_k) in [(256, 24, 128), (128, 17, 32)]:
        xin = (torch.randn(k, n) * 3).to(torch.bfloat16)
        q, sf = rmath.per_channel_cast_to_fp8(xin, use_ue8m0=True, gran_k=gran_k)
        out['quant'].append({'kind': 'channel', 'x': xin, 'use_ue8m0': True, 'gran_k': gran_k,
                             'q': q.view(torch.uint8), 'sf': sf})

    # packed UE8M0 wire format (tests/test_layout.py:20-42), incl. unaligned mn / k and batches
    for (b, mn, sf_k) in [(1, 5, 1), (1, 128, 56), (1, 130, 57), (2, 33, 14), (4, 64, 3), (1, 4097, 2)]:
        e = torch.randint(1, 255, (b, mn, sf_k), dtype=torch.int32)
        sf = (e << 23).view(torch.float32)
        sf_in = sf[0] if b == 1 else sf
        packed = ref_layout.get_mn_major_tma_aligned_packed_ue8m0_tensor_torch_impl(sf_in)
        out['pack'].append({'sf': sf_in, 'packed': packed.clone(memory_format=torch.preserve_format),
                            'shape': tuple(packed.shape), 'stride': tuple(packed.stride()),
                            'dense': torch.empty(packed.shape, dtype=torch.int32).copy_(packed)})

    for _ in range(4):
        a, b_ = torch.randn(64, 64), torch.randn(64, 64)
        out['calc_diff'].append({'x': a, 'y': a + 0.01 * b_, 'd': float(calc_diff(a, a + 0.01 * b_))})
    out['calc_diff'].append({'x': torch.zeros(4), 'y': torch.zeros(4), 'd': float(calc_diff(torch.zeros(4), torch.zeros(4)))})

    import store
    for path in store.save(out, HERE, 'cpu_golden'):
        print('wrote', path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
