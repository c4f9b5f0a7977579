"""Generate GPU golden vectors WITH THE REFERENCE'S OWN SM100 KERNEL (run on a B200 under gpurun; needs the
reference install oracle/_ref built by oracle/build_ref.sh; nothing here touches /root/reference at run time).

For a few small seeded problems it stores the FP8 operands, scale factors and the output of the unmodified
reference (`deep_gemm.fp8_gemm_nt`, `m_grouped_fp8_gemm_nt_masked`, `m_grouped_fp8_gemm_nt_contiguous`).
Output: tests/golden/gpu_golden.*.pt (tests/golden/store.py), or under the directory given as the first argument.
"""
import os
import random
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))


def main():
    os.environ.setdefault('DG_JIT_CACHE_DIR', '/tmp/dg_ref_cache')
    os.environ.setdefault('CUDA_HOME', '/usr/local/cuda')
    sys.path.insert(0, os.path.join(REPO, 'oracle', '_ref'))
    import deep_gemm as ref
    from deep_gemm.utils import per_block_cast_to_fp8, per_token_cast_to_fp8
    assert 'oracle/_ref' in ref.__file__
    torch.manual_seed(1234)
    random.seed(1234)
    out = {'dense': [], 'masked': [], 'contiguous': [], 'reference_version': ref.__version__}

    def u8(t):
        return t.view(torch.uint8).cpu()

    for (m, n, k, dtype, acc) in [(128, 128, 128, torch.bfloat16, False), (64, 256, 512, torch.bfloat16, False),
                                  (200, 384, 1024, torch.float32, False), (33, 136, 640, torch.bfloat16, True),
                                  (96, 256, 384, torch.float32, True), (1, 576, 768, torch.bfloat16, False)]:
        a = torch.randn((m, k), device='cuda', dtype=torch.bfloat16)
        b = torch.randn((n, k), device='cuda', dtype=torch.bfloat16)
        qa, qb = per_token_cast_to_fp8(a, True), per_block_cast_to_fp8(b, True)
        c = (torch.randn((m, n), device='cuda') * 8).to(dtype) if acc else None
        d = c.clone() if acc else torch.empty((m, n), device='cuda', dtype=dtype)
        ref.fp8_gemm_nt(qa, qb, d, c=d if acc else None)
        torch.cuda.synchronize()
        out['dense'].append({'name': f'dense_{m}x{n}x{k}_{dtype}_{acc}', 'a': u8(qa[0]), 'sfa': qa[1].cpu(), 'b': u8(qb[0]),
                             'sfb': qb[1].cpu(), 'c': None if c is None else c.cpu(), 'd': d.cpu()})

    # NOTE: M_max must be a multiple of the reference's BLOCK_M (128 here): its masked kernel stores whole tiles, so with
    # M_max=96 a tile of group g spills over the first rows of group g+1 (SURVEY Appendix E pitfall 1) -- not golden.
    g, m_max, n, k = 4, 128, 256, 512
    a = torch.randn((g, m_max, k), device='cuda', dtype=torch.bfloat16)
    b = torch.randn((g, n, k), device='cuda', dtype=torch.bfloat16)
    qa_l = [per_token_cast_to_fp8(a[i], True) for i in range(g)]
    qb_l = [per_block_cast_to_fp8(b[i], True) for i in range(g)]
    qa = (torch.stack([x[0] for x in qa_l]), torch.stack([x[1] for x in qa_l]))
    qb = (torch.stack([x[0] for x in qb_l]), torch.stack([x[1] for x in qb_l]))
    masked_m = torch.tensor([17, 128, 0, 50], device='cuda', dtype=torch.int32)
    d = torch.zeros((g, m_max, n), device='cuda', dtype=torch.bfloat16)
    ref.m_grouped_fp8_gemm_nt_masked(qa, qb, d, masked_m, 48)
    torch.cuda.synchronize()
    out['masked'].append({'name': 'masked_4x128x256x512', 'a': u8(qa[0]), 'sfa': qa[1].cpu(), 'b': u8(qb[0]), 'sfb': qb[1].cpu(),
                          'masked_m': masked_m.cpu(), 'expected_m': 48, 'd': d.cpu()})

    for psum in (False, True):
        alignment = 128
        ref.set_mk_alignment_for_contiguous_layout(alignment)
        ms = [70, 128, 5]
        aligned = [(x + alignment - 1) // alignment * alignment for x in ms]
        m = sum(aligned)
        a = torch.randn((m, k), device='cuda', dtype=torch.bfloat16)
        layout = torch.empty(len(ms) if psum else m, device='cuda', dtype=torch.int32)
        valid = torch.zeros(m, dtype=torch.bool)
        s = 0
        for i, (mi, ai) in enumerate(zip(ms, aligned)):
            if psum:
                layout[i] = s + mi
            else:
                layout[s:s + mi] = i
                layout[s + mi:s + ai] = -1
            a[s + mi:s + ai] = 0
            valid[s:s + mi] = True
            s += ai
        qa = per_token_cast_to_fp8(a, True)
        qb3 = (qb[0][:3].contiguous(), qb[1][:3].contiguous())
        d = torch.zeros((m, n), device='cuda', dtype=torch.bfloat16)
        ref.m_grouped_fp8_gemm_nt_contiguous(qa, qb3, d, layout, use_psum_layout=psum)
        torch.cuda.synchronize()
        out['contiguous'].append({'name': f'contiguous_psum{psum}', 'a': u8(qa[0]), 'sfa': qa[1].cpu(), 'b': u8(qb3[0]),
                                  'sfb': qb3[1].cpu(), 'layout': layout.cpu(), 'psum': psum, 'alignment': alignment,
                                  'valid': valid, 'd': d.cpu()})

    # MN-major operands (fp8_gemm_tn: A [K,M], B [K,N]) and the K-grouped weight gradient
    out['dense_tn'], out['k_grouped'] = [], []
    for (m, n, k) in [(128, 256, 384), (192, 128, 512)]:
        a = torch.randn((m, k), device='cuda', dtype=torch.bfloat16)
        b = torch.randn((n, k), device='cuda', dtype=torch.bfloat16)
        qa, qb = per_token_cast_to_fp8(a, True), per_block_cast_to_fp8(b, True)
        a_t = (qa[0].t().contiguous(), qa[1].t().contiguous())
        b_t = (qb[0].t().contiguous(), qb[1].t().contiguous())
        d = torch.empty((m, n), device='cuda', dtype=torch.bfloat16)
        ref.fp8_gemm_tn(a_t, b_t, d)
        torch.cuda.synchronize()
        out['dense_tn'].append({'name': f'tn_{m}x{n}x{k}', 'a_t': u8(a_t[0]), 'sfa_t': a_t[1].cpu(), 'b_t': u8(b_t[0]),
                                'sfb_t': b_t[1].cpu(), 'd': d.cpu()})
    from deep_gemm.utils import per_channel_cast_to_fp8
    for gran_k, k_alignment in ((128, 128), (32, 32)):
        ref.set_mk_alignment_for_contiguous_layout(k_alignment)
        ks = [k_alignment * 3, 0, k_alignment * 1, k_alignment * 5]
        m, n = 256, 128
        a = torch.randn((sum(ks), m), device='cuda', dtype=torch.bfloat16)
        b = torch.randn((sum(ks), n), device='cuda', dtype=torch.bfloat16)
        qa_l, qb_l, sa_l, sb_l, pos = [], [], [], [], 0
        for kk in ks:
            if kk == 0:
                continue
            pad = (kk + gran_k - 1) // gran_k * gran_k
            xa = torch.zeros((pad, m), device='cuda', dtype=torch.bfloat16)
            xb = torch.zeros((pad, n), device='cuda', dtype=torch.bfloat16)
            xa[:kk], xb[:kk] = a[pos:pos + kk], b[pos:pos + kk]
            qa_, sa_ = per_channel_cast_to_fp8(xa, use_ue8m0=True, gran_k=gran_k)
            qb_, sb_ = per_channel_cast_to_fp8(xb, use_ue8m0=True, gran_k=gran_k)
            qa_l.append(qa_[:kk]), qb_l.append(qb_[:kk]), sa_l.append(sa_), sb_l.append(sb_)
            pos += kk
        a8, b8, sfa, sfb = torch.cat(qa_l), torch.cat(qb_l), torch.cat(sa_l), torch.cat(sb_l)
        c = torch.randn((len(ks), m, n), device='cuda') * 8
        d = c.clone()
        ref.k_grouped_fp8_gemm_tn_contiguous((a8, sfa), (b8, sfb), d, ks, torch.tensor(ks, device='cuda', dtype=torch.int32),
                                             c=d, recipe=(1, 1, gran_k))
        torch.cuda.synchronize()
        out['k_grouped'].append({'name': f'k_grouped_g{gran_k}', 'a': u8(a8), 'sfa': sfa.cpu(), 'b': u8(b8), 'sfb': sfb.cpu(),
                                 'c': c.cpu(), 'd': d.cpu(), 'ks': ks, 'gran_k': gran_k, 'k_alignment': k_alignment})
    ref.set_mk_alignment_for_contiguous_layout(128)

    import store
    out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(out_dir, exist_ok=True)
    for path in store.save(out, out_dir, 'gpu_golden'):
        print('wrote', path, os.path.getsize(path))


if __name__ == '__main__':
    main()
