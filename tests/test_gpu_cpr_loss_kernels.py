"""The three kernels of the CPR training loss, called directly and compared with a float64 reference of the same operation on the
logit map, at every class-count regime they have:

  bag_mil_fwd_kernel            fused ring-bag gather + MIL forward (online softmax); 320 threads = ceil(N/4) class groups x sample slices
  cpr_loss_bwd_tile_kernel      deterministic backward, one CTA of 64 * LD/32 threads per 8x8 map tile (LD = 2 * ceil8(N) <= 160)
  cpr_loss_bwd_scatter_kernel   default backward, one CTA per bag, fp32 vector atomics into the map

and a head-level sweep (CPRHead.loss + backward in the three backward modes) at class counts whose logit rows are 32 to 128 wide.
The reference is written from the oracle's building blocks (grid_sample sampling, point validity, MIL bag probability, gfocal loss) and
differentiated by float64 autograd; the kernels are compared with it, never with each other."""
import os

import numpy as np
import pytest
import torch

from oracle import cpr as ocpr, synth
from tests.helpers import assert_close, oracle_cfg, scale_rel_err

pytestmark = pytest.mark.gpu

EPS = 1e-6
STRIDE = 8.0
S_MIL, S_GT, S_NEG = 0.37, 0.21, 0.53          # scalar multipliers of the three loss terms (upstream gradient x weight / normaliser)
PROB_BOUND = 1e-4                              # |prob| <= 1: a top-1 decision closer than this may legitimately differ from float64


# ------------------------------------------------------------------------------------------------------------------------------------
# float64 reference (CPU)
# ------------------------------------------------------------------------------------------------------------------------------------
def loss_reference(lmap, centers, labels, bag_img, img_ptr, offsets, pad_hw, stride, N, NP, eps, s_mil, s_gt, s_neg, neg_mask):
    """The CPR loss on a (B,H,W,LD) logit map [cls (0..N) pad | ins (NP..NP+N) pad] in float64:

        total = s_mil * sum_g lw_g * gfocal(prob_g, onehot_g)                    MIL bag loss (ring bags, centre sample last)
              + s_gt  * sum_g valid_g,centre * gfocal(sigmoid(cls_g,centre), onehot_g)
              + s_neg * sum_cells,c<N neg_mask * gfocal(sigmoid(lmap[cell, c]), 0)

    s_gt / s_neg None drop their term.  The sample points are formed in float32 (offset + centre, as the kernels do) and only then
    cast to float64 for grid_sample.  Returns the forward quantities the kernels produce and d(bag terms)/d lmap, d(neg term)/d lmap."""
    B, H, W, LD = lmap.shape
    G, K = centers.shape[0], offsets.shape[0]
    lm = lmap.double().requires_grad_(True)
    pts = offsets[None, :, :] + centers[:, None, :]                                  # float32 (G,K,2)
    parts, valid = [], torch.zeros(G, K, dtype=torch.bool)
    for b in range(B):
        lo, hi = int(img_ptr[b]), int(img_ptr[b + 1])
        assert bool((bag_img[lo:hi] == b).all())
        if hi > lo:
            parts.append(ocpr.sample_point_feat(lm[b].permute(2, 0, 1)[None], pts[lo:hi].double(), stride))
            valid[lo:hi] = ocpr.point_valid(pts[lo:hi], int(pad_hw[b, 0]), int(pad_hw[b, 1]))
    bl = torch.cat(parts)                                                            # (G,K,LD)
    w = valid.double()
    cls, ins = bl[..., :N], bl[..., NP:NP + N]
    prob = ocpr.mil_bag_prob(cls.sigmoid(), ins, w[..., None])                       # (G,N)
    lw = (w.sum(dim=1) > 0).double()
    onehot = torch.zeros(G, N, dtype=torch.float64)
    onehot[torch.arange(G), labels.long()] = 1
    mil = ocpr.gfocal_loss(prob, onehot, lw[:, None], eps)                           # (G,)
    total = s_mil * mil.sum()
    if s_gt is not None:
        total = total + s_gt * ocpr.gfocal_loss(cls[:, K - 1].sigmoid(), onehot, w[:, K - 1:K], eps).sum()
    grad_bags, = torch.autograd.grad(total, lm, retain_graph=s_neg is not None)
    grad_neg = torch.zeros_like(grad_bags)
    if s_neg is not None:
        negp = lm[..., :N].sigmoid().reshape(-1, N)
        neg = ocpr.gfocal_loss(negp, torch.zeros_like(negp), neg_mask.reshape(-1, N).double(), eps).sum()
        grad_neg, = torch.autograd.grad(s_neg * neg, lm)
    with torch.no_grad():
        m = ins.max(dim=1)[0]                                                        # (G,N): max over ALL samples (softmax shift)
        e = (ins - m[:, None]).exp()
        Z, T = e.sum(dim=1), (e * w[..., None]).sum(dim=1)
        inv_t = torch.where(T / Z >= 1e-12, 1.0 / T, torch.zeros_like(T))           # 0 where F.normalize's clamp is active
        top = prob.argmax(dim=1)
        own = prob[torch.arange(G), labels.long()]
        other = prob.clone()
        other[torch.arange(G), labels.long()] = -1.0
        margin = (own - other.max(dim=1)[0]).abs() if N > 1 else torch.full((G,), float('inf'), dtype=torch.float64)
        # map cells some bag sample reaches (bilinear taps, dilated by one cell): everywhere else only the neg term may appear
        p64 = pts.double() / stride
        ix = p64[..., 0].clamp(0, W - 1).floor().long()
        iy = p64[..., 1].clamp(0, H - 1).floor().long()
        reached = torch.zeros(B, H, W, dtype=torch.bool)
        bi = bag_img.long()[:, None].expand(G, K)
        for dy in (0, 1):
            for dx in (0, 1):
                reached[bi, (iy + dy).clamp(max=H - 1), (ix + dx).clamp(max=W - 1)] = True
        reached = torch.nn.functional.max_pool2d(reached[:, None].double(), 3, 1, 1)[:, 0] > 0
    return dict(bl=bl.detach(), valid=valid, prob=prob.detach(), loss_sum=mil.sum().detach(), n_weighted=lw.sum(),
                hits=(top == labels.long()), margin=margin.detach(), max_ins=m.detach(), inv_t=inv_t.detach(), lw=lw,
                grad_bags=grad_bags, grad_neg=grad_neg, reached=reached)


# ------------------------------------------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------------------------------------------
def _case(cid, N, radius, hw, images, pad=None, gt=True, neg=True, seed=0):
    return pytest.param(dict(N=N, radius=radius, hw=hw, images=images, pad=pad, gt=gt, neg=neg, seed=seed), id=cid)


# image specs: ('rand', n) uniform in the pad area; ('tile', n) centres inside the first 8x8 tile (dense overlap: the 512-record buffer
# of the tile kernel flushes); ('edges', n) on the right and bottom pad edges (clamped east / south taps, weight 0); ('corners',) a centre
# at (0,0), centres at the pad border (pw - 1e-3, ph - 1e-3) and a bag whose samples all lie outside the pad (label weight 0, 1/T = 0)
CASES = [
    _case('n1_r2_corners', 1, 2, (24, 32), [[('corners',), ('rand', 20)]]),
    _case('n7_r5_edges_odd_pad', 7, 5, (37, 53), [[('edges', 12), ('rand', 30)], [('rand', 25), ('corners',)]], pad=(37 * 8 - 5, 53 * 8 - 11)),
    _case('n10_r5_dense', 10, 5, (37, 53), [[('tile', 40), ('rand', 60), ('corners',)]]),
    _case('n10_r2_1100gts', 10, 2, (40, 60), [[('rand', 1100)], [('rand', 30), ('edges', 6)]]),
    _case('n10_r2_narrow', 10, 2, (20, 6), [[('rand', 25), ('corners',)]]),
    _case('n16_r8_corners', 16, 8, (30, 40), [[('corners',), ('tile', 20), ('rand', 40)]]),
    _case('n16_r9', 16, 9, (30, 40), [[('tile', 10), ('rand', 30), ('corners',)]]),
    _case('n20_r1_dense', 20, 1, (37, 53), [[('tile', 60), ('rand', 200)]]),
    _case('n32_r5_dense', 32, 5, (37, 53), [[('tile', 40), ('rand', 40), ('edges', 8)]]),
    _case('n32_r5_no_gt_no_neg', 32, 5, (24, 40), [[('tile', 30), ('rand', 30), ('corners',)]], gt=False, neg=False),
    _case('n33_r2', 33, 2, (24, 40), [[('tile', 20), ('rand', 40), ('corners',)]]),
    _case('n48_r5_dense_empty_image', 48, 5, (37, 53), [[('tile', 40), ('rand', 50)], [], [('rand', 20), ('corners',)]]),
    _case('n64_r8_dense', 64, 8, (32, 40), [[('tile', 30), ('rand', 40), ('edges', 6)]]),
    _case('n80_r5_dense_no_neg', 80, 5, (37, 53), [[('tile', 40), ('rand', 40), ('corners',)]], neg=False),
    _case('n80_r1_narrow', 80, 1, (12, 5), [[('rand', 15), ('corners',)], [('rand', 10)]]),
    _case('n128_r9', 128, 9, (30, 40), [[('tile', 20), ('rand', 30), ('corners',)]]),
]


def make_case(c):
    """seeded CPU inputs of one case: a (B,H,W,LD) logit map with zero pad channels (as the head builds it), GT centres / labels in
    CSR order, the ring offsets (centre last) and the pad shapes."""
    from pointtinybenchmark_b200 import ops
    N = c['N']
    NP = (N + 7) // 8 * 8
    LD = 2 * NP
    H, W = c['hw']
    B = len(c['images'])
    ph, pw = c['pad'] or (int(H * STRIDE), int(W * STRIDE))
    rng = np.random.default_rng(1000 + 17 * N + c['radius'] + c['seed'])
    centers, lens = [], []
    for spec in c['images']:
        pts = [np.zeros((0, 2))]
        for item in spec:
            kind = item[0]
            if kind == 'rand':
                pts.append(rng.uniform([0, 0], [pw, ph], (item[1], 2)))
            elif kind == 'tile':
                pts.append(rng.uniform(0.5 * STRIDE, 7.5 * STRIDE, (item[1], 2)))
            elif kind == 'edges':
                n = item[1]
                right = np.stack([pw - rng.uniform(0, 3, n), rng.uniform(0, ph, n)], 1)
                bottom = np.stack([rng.uniform(0, pw, n), ph - rng.uniform(0, 3, n)], 1)
                pts += [right, bottom]
            else:
                pts.append(np.array([[0.0, 0.0], [pw - 1e-3, ph - 1e-3], [pw - 1e-3, 0.0], [0.0, ph - 1e-3], [-900.0, -900.0]]))
        p = np.concatenate(pts)
        centers.append(p)
        lens.append(len(p))
    centers = torch.from_numpy(np.concatenate(centers)).float().contiguous()
    G = centers.shape[0]
    labels = torch.from_numpy(rng.integers(0, N, G)).int()
    bag_img = torch.from_numpy(np.repeat(np.arange(B), lens)).int()
    img_ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)])).int()
    pad_hw = torch.tensor([[ph, pw]] * B, dtype=torch.int32)
    lmap = torch.zeros(B, H, W, LD)
    lmap[..., :N] = torch.from_numpy(rng.normal(-1.5, 1.5, (B, H, W, N))).float()
    lmap[..., NP:NP + N] = torch.from_numpy(rng.normal(0.0, 1.5, (B, H, W, N))).float()
    offsets = ops.circle_offsets(c['radius'], STRIDE)
    return dict(N=N, NP=NP, LD=LD, B=B, H=H, W=W, G=G, K=offsets.shape[0], lmap=lmap, centers=centers, labels=labels, bag_img=bag_img,
                img_ptr=img_ptr, pad_hw=pad_hw, offsets=offsets)


def _tile_kernel_accepts(x):
    return x['LD'] % 32 == 0 and x['LD'] <= 160 and x['K'] <= 320


@pytest.fixture(scope='module')
def ops():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from pointtinybenchmark_b200 import ops as _ops
    return _ops


def _pad_cols(x):
    N, NP, LD = x['N'], x['NP'], x['LD']
    return torch.cat([torch.arange(N, NP), torch.arange(NP + N, LD)]).long()


def _check_map_grad(what, got, ref, x, reached, exact_outside):
    """pad channels exactly 0; everywhere within the gradient tolerance of float64; unreached cells exactly `exact_outside`."""
    got = got.cpu()
    pc = _pad_cols(x)
    assert bool((got[..., pc] == 0).all()), f'{what}: pad channels are not 0'
    e = assert_close(got, ref, 2e-4, what)
    far = ~reached
    if bool(far.any()):
        want = exact_outside[far]
        mism = (got[far] != want) & ~torch.isnan(want)
        assert not bool(mism.any()), f'{what}: {int(mism.sum())} values on cells no bag reaches are not exactly the expected ones'
    return e


@pytest.mark.parametrize('case', CASES)
def test_loss_kernels_against_float64(ops, case):
    x = make_case(case)
    N, NP, LD, B, H, W, G, K = (x[k] for k in ('N', 'NP', 'LD', 'B', 'H', 'W', 'G', 'K'))
    dev = torch.device('cuda:0')
    d = {k: x[k].to(dev).contiguous() for k in ('lmap', 'centers', 'labels', 'bag_img', 'img_ptr', 'pad_hw', 'offsets')}
    nm = ops.neg_mask(B, H, W, STRIDE, d['pad_hw'], d['centers'], d['labels'], d['img_ptr'], STRIDE * case['radius'], N, True, as_bool=False)
    ref = loss_reference(x['lmap'], x['centers'], x['labels'], x['bag_img'], x['img_ptr'], x['offsets'], x['pad_hw'], STRIDE, N, NP, EPS,
                         S_MIL, S_GT if case['gt'] else None, S_NEG if case['neg'] else None, nm.cpu())

    # ---- fused gather + MIL forward
    bl, weight, bag_prob, loss_sum, stats, mt, lw = ops.bag_mil_fwd(d['lmap'], N, NP, d['centers'], d['bag_img'], d['offsets'], STRIDE,
                                                                      d['pad_hw'], d['labels'], EPS)
    torch.cuda.synchronize()
    blc = bl.cpu()
    assert torch.equal(weight.cpu(), ref['valid'].float()), 'sample validity'
    assert torch.equal(lw.cpu(), ref['lw'].float()), 'label weight'
    assert bool((blc[..., _pad_cols(x)] == 0).all()), 'pad columns of the bag logits are not 0'
    bound = float(x['lmap'].abs().max()) * 2.0 ** -24 * (16 * max(H, W) + 64)       # fp32 sample coordinates + bilinear rounding
    ebl = float((blc.double() - ref['bl']).abs().max())
    assert ebl <= bound, f'bag logits: max |err| {ebl:.3e} > fp32 bilinear bound {bound:.3e}'
    assert torch.equal(mt[..., 0].cpu(), blc[:, :, NP:NP + N].max(dim=1)[0]), 'max ins is not the max of the written bag logits'
    e_m = assert_close(mt[..., 0], ref['max_ins'], 1e-4, 'max ins')
    e_t = assert_close(mt[..., 1], ref['inv_t'], 1e-4, '1/T')
    assert bool((mt[..., 1].cpu()[ref['lw'] == 0] == 0).all()), '1/T must be 0 for a bag without a valid sample'
    e_p = assert_close(bag_prob, ref['prob'], 1e-4, 'bag probability')
    e_l = assert_close(loss_sum, ref['loss_sum'].reshape(1), 1e-4, 'MIL loss sum')
    st = stats.cpu()
    assert float(st[0]) == float(ref['n_weighted']), 'bags with weight'
    hits = (bag_prob.cpu().argmax(dim=1) == x['labels'].long())
    assert float(st[1]) == float(hits.sum()), 'top-1 hits != the hits of the written bag probabilities'
    sure = ref['margin'] > PROB_BOUND
    assert torch.equal(hits[sure], ref['hits'][sure]), 'top-1 decision with a float64 margin above the bound differs'

    # ---- backward: terms as the head passes them
    f1 = lambda v: torch.tensor([v], dtype=torch.float32, device=dev)
    wc = weight[:, K - 1].contiguous()
    kw = dict(scale_mil=f1(S_MIL), scale_gt=f1(S_GT) if case['gt'] else None, valid_center=wc if case['gt'] else None)
    grad_bags, grad_neg = ref['grad_bags'], ref['grad_neg']
    # values that must come out exactly on cells no bag reaches: 0, except the neg term on masked class channels (NaN: not exact)
    outside = torch.zeros(B, H, W, LD, dtype=torch.float64)
    if case['neg']:
        outside[..., :N][nm.cpu().bool()] = float('nan')
    errs = {}
    if _tile_kernel_accepts(x):
        neg_kw = dict(logit_map=d['lmap'], neg_mask=nm, scale_neg=f1(S_NEG)) if case['neg'] else {}
        runs = []
        for _ in range(2):
            out = torch.full((B, H, W, LD), float('nan'), device=dev)
            ops.cpr_loss_bwd_map(bl, weight, mt, bag_prob, lw, d['labels'], d['centers'], d['img_ptr'], d['offsets'], (B, H, W, LD), N, NP,
                                 STRIDE, ops.offsets_reach(d['offsets']), EPS, out=out, **kw, **neg_kw)
            runs.append(out)
        assert torch.equal(runs[0], runs[1]), 'cpr_loss_bwd_map differs between two runs'
        errs['tiles'] = _check_map_grad('cpr_loss_bwd_map', runs[0], grad_bags + grad_neg, x, ref['reached'], outside)
    else:
        with pytest.raises(RuntimeError, match='ptb_cpr_loss_bwd_map'):
            ops.cpr_loss_bwd_map(bl, weight, mt, bag_prob, lw, d['labels'], d['centers'], d['img_ptr'], d['offsets'], (B, H, W, LD), N, NP,
                                 STRIDE, ops.offsets_reach(d['offsets']), EPS, **kw)
    gm = torch.zeros(B, H, W, LD, device=dev)
    ops.cpr_loss_bwd_scatter(bl, weight, mt, bag_prob, lw, d['labels'], d['centers'], d['bag_img'], d['offsets'], gm, N, NP, STRIDE, EPS,
                             **kw)
    errs['scatter'] = _check_map_grad('cpr_loss_bwd_scatter', gm, grad_bags, x, ref['reached'], torch.zeros_like(outside))
    print(f'[loss kernels N={N} K={K} LD={LD} G={G} {H}x{W}] bl {ebl:.1e} (bound {bound:.1e}), max ins {e_m:.1e}, 1/T {e_t:.1e}, '
          f'prob {e_p:.1e}, loss {e_l:.1e}, grad ' + ', '.join(f'{k} {v:.1e}' for k, v in errs.items()) +
          f'; top-1 within bound {int((~sure).sum())}/{G}')


# ------------------------------------------------------------------------------------------------------------------------------------
# head level: CPRHead.loss + backward in each backward mode vs oracle.cpr.cpr_loss (float64 autograd)
# ------------------------------------------------------------------------------------------------------------------------------------
_ORACLE = {}


def _oracle(inp, N):
    if N not in _ORACLE:
        cfg = oracle_cfg(inp['cfgd'])
        fo = inp['cls_feat'].double().requires_grad_(True)
        wo = {k: v.double().requires_grad_(True) for k, v in inp['weights'].items()}
        ol, aux = ocpr.cpr_loss(fo, wo, inp['gt_bboxes'], inp['gt_labels'], inp['img_metas'], cfg, return_all=True)
        sum(v for k, v in ol.items() if 'loss' in k).backward()
        _ORACLE[N] = ({k: v.detach() for k, v in ol.items()}, fo.grad, {k: v.grad for k, v in wo.items()}, aux['bag_prob'].detach())
    return _ORACLE[N]


@pytest.mark.parametrize('mode', ['tiles', 'scatter', 'staged'])
@pytest.mark.parametrize('N', [10, 32, 48, 64])
def test_head_loss_grads_by_class_count(ops, monkeypatch, N, mode):
    from pointtinybenchmark_b200 import cpr_head  # noqa: F401  (registers the head)
    from pointtinybenchmark_b200.registry import build_head
    from tests.test_gpu_cpr_head import head_cfg
    dev = torch.device('cuda:0')
    inp = synth.cpr_inputs('lite', 2024, num_classes=N)
    head = build_head(head_cfg(inp['cfgd'])).to(dev)
    sd = head.state_dict()
    sd.update(inp['weights'])
    head.load_state_dict(sd, strict=True)
    gtb = [b.to(dev) for b in inp['gt_bboxes']]
    gtl = [l.to(dev) for l in inp['gt_labels']]
    calls = {'cpr_loss_bwd_map': 0, 'cpr_loss_bwd_scatter': 0}
    for name in calls:
        fn = getattr(ops, name)

        def spy(*a, _fn=fn, _name=name, **k):
            calls[_name] += 1
            return _fn(*a, **k)
        monkeypatch.setattr(ops, name, spy)

    def run(env):
        if env is not None:
            os.environ['PTB_LOSS_BWD'] = env
        try:
            head.zero_grad(set_to_none=True)
            feat = inp['cls_feat'].to(dev).contiguous(memory_format=torch.channels_last).requires_grad_(True)
            losses = head.loss([feat], [feat], gtb, gtl, inp['img_metas'])
            sum(v for k, v in losses.items() if 'loss' in k).backward()
            return losses, [feat.grad.clone()] + [p.grad.clone() for p in (head.cls_out.weight, head.cls_out.bias, head.ins_out.weight,
                                                                            head.ins_out.bias)]
        finally:
            os.environ.pop('PTB_LOSS_BWD', None)

    losses, grads = run(mode)
    want = {'tiles': (1, 0), 'scatter': (0, 1), 'staged': (0, 0)}[mode]
    assert (calls['cpr_loss_bwd_map'], calls['cpr_loss_bwd_scatter']) == want, f'mode {mode} ran {calls}'
    if mode == 'tiles':
        # torch.use_deterministic_algorithms(True) must select the tile kernel too, and give the same bits
        torch.use_deterministic_algorithms(True)
        try:
            _, again = run(None)
        finally:
            torch.use_deterministic_algorithms(False)
        assert calls['cpr_loss_bwd_map'] == 2 and calls['cpr_loss_bwd_scatter'] == 0, f'deterministic mode ran {calls}'
        assert all(torch.equal(a, b) for a, b in zip(grads, again)), 'deterministic mode: gradients differ between two runs'
    ol, fgrad, wgrad, bag_prob = _oracle(inp, N)
    for k in ('gt_loss', 'pos_loss', 'neg_loss'):
        assert_close(losses[k].reshape(-1), ol[k].reshape(-1), 1e-4, f'N={N} {mode} {k}')
    # bag_acc counts top-1 hits: a bag whose float64 decision margin is inside the bound may legitimately flip
    labels = torch.cat(inp['gt_labels'])
    p = bag_prob.clone()
    own = p[torch.arange(len(labels)), labels].clone()
    p[torch.arange(len(labels)), labels] = -1.0
    unsure = int(((own - p.max(dim=1)[0]).abs() <= PROB_BOUND).sum())
    dacc = abs(float(losses['bag_acc'].reshape(-1)[0]) - float(ol['bag_acc'].reshape(-1)[0]))
    assert dacc <= unsure * 100.0 / len(labels) + 1e-3, f'N={N} {mode} bag_acc differs by {dacc} ({unsure} undecided bags)'
    e = assert_close(grads[0], fgrad, 2e-4, f'N={N} {mode} d loss / d feature map')
    e2 = assert_close(grads[1], wgrad['cls_out.weight'], 2e-4, f'N={N} {mode} dW cls')
    e3 = assert_close(grads[3], wgrad['ins_out.weight'], 2e-4, f'N={N} {mode} dW ins')
    e4 = assert_close(grads[2], wgrad['cls_out.bias'], 2e-4, f'N={N} {mode} db cls')
    # softmax over the bag is shift invariant: the ins bias gradient is analytically zero (fp noise on both sides)
    assert float((grads[4].cpu().double() - wgrad['ins_out.bias']).abs().max()) <= 1e-5 * float(wgrad['ins_out.weight'].abs().max())
    print(f'[head N={N} {mode}] feat {e:.1e}, dW cls {e2:.1e}, dW ins {e3:.1e}, db cls {e4:.1e}; '
          f'losses ' + ', '.join(f'{k} {scale_rel_err(losses[k].reshape(-1), ol[k].reshape(-1)):.1e}' for k in ('gt_loss', 'pos_loss', 'neg_loss')))
