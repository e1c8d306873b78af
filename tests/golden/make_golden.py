#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference,
anuragranj/cc @ 2b4e362) on CPU fp32 in the build container.

The reference is Python and cannot travel to the GPU box, so its outputs (and autograd
gradients) on seeded synthetic inputs are frozen here.  Run:  python tests/golden/make_golden.py
Stubs (reference cannot import/run without them, SURVEY.md F11):
  * spatial_correlation_sampler -> oracle.nets.spatial_correlation_sample (third-party op absent
    from the tree; that boundary stays "parity unpinned")
  * torch.Tensor.cuda / Module.cuda -> no-op (Back2Future calls .cuda() in __init__/warp)
"""
import os
import sys
import types
import warnings
import zlib
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = os.environ.get('CC_REFERENCE', '/root/reference')
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)
warnings.filterwarnings('ignore')

from cc_b200 import synth            # noqa: E402
from oracle import nets as onets     # noqa: E402

stub = types.ModuleType('spatial_correlation_sampler')
stub.spatial_correlation_sample = lambda a, b, kernel_size=1, patch_size=9, stride=1: \
    onets.spatial_correlation_sample(a, b, patch_size)
sys.modules['spatial_correlation_sampler'] = stub
torch.Tensor.cuda = lambda self, *a, **k: self
torch.nn.Module.cuda = lambda self, *a, **k: self

import inverse_warp as RW            # noqa: E402
import loss_functions as RL          # noqa: E402
import ssim as RS                    # noqa: E402
import models as RM                  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
torch.manual_seed(0)
torch.set_num_threads(8)


def npy(t):
    return t.detach().cpu().numpy()


PART_BYTES = 900 * 1024      # no fixture file over 1 MB: a larger fixture is stored as name.npz, name.1.npz, ...


def save(name, d):
    arrs = {k: (npy(v) if torch.is_tensor(v) else np.asarray(v)) for k, v in d.items()}
    write_parts(name, arrs)
    print(name, len(arrs), 'arrays')


def part_path(name, i):
    return os.path.join(OUT, name + ('.%d' % i if i else '') + '.npz')


def write_parts(name, arrs):
    """Arrays in key order, cut into parts of about PART_BYTES (zlib estimate of the deflated members, which leaves room
    for the npz headers under 1 MB); tests/util.golden() joins the parts."""
    parts, size = [{}], 0
    for k, a in arrs.items():
        n = len(zlib.compress(a.tobytes()))
        if n > PART_BYTES:
            raise ValueError('%s: array %s deflates to %d bytes, more than one part holds; store a strided sample '
                             '(compact())' % (name, k, n))
        if parts[-1] and size + n > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = a
        size += n
    for i, p in enumerate(parts):
        np.savez_compressed(part_path(name, i), **p)
    i = len(parts)
    while os.path.exists(part_path(name, i)):          # parts left over from a larger earlier run
        os.remove(part_path(name, i))
        i += 1


def compact(g, limit=40000, stride=61):
    """Big gradient tensors are frozen as a strided subsample (key suffix '@61')."""
    if g.numel() <= limit:
        return '', g
    return '@%d' % stride, g.flatten()[::stride]


def leaf(t):
    return t.detach().clone().requires_grad_(True)


def wts(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


# --------------------------------------------------------------------------- A. warp layer
def gen_warp():
    B, H, W = 2, 24, 40
    s = synth.sample(B, H, W, seed=10, nlevels=1)
    d = dict(B=B, H=H, W=W)
    img = s['refs'][0]
    depth = leaf(s['depth'][0][:, 0])
    pose = leaf(s['pose'][:, 0])
    K, Kinv = s['K'], s['Kinv']
    for pm in ('zeros', 'border'):
        out = RW.inverse_warp(img, depth, pose, K, Kinv, 'euler', pm)
        wt = wts(out.shape, 1)
        gd, gp = torch.autograd.grad((out * wt).sum(), [depth, pose])
        d.update({f'iw_{pm}_out': out, f'iw_{pm}_gdepth': gd, f'iw_{pm}_gpose': gp})
    d['iw_wt'] = wts(out.shape, 1)
    outq = RW.inverse_warp(img, depth, pose, K, Kinv, 'quat', 'zeros')
    d['iw_quat_out'] = outq
    flow = leaf(s['flow_fwd'][0])
    imgl = leaf(img)
    fw = RW.flow_warp(imgl, flow)
    gf, gi = torch.autograd.grad((fw * d['iw_wt']).sum(), [flow, imgl])
    d.update(fw_out=fw, fw_gflow=gf, fw_gimg=gi)
    p2f = RW.pose2flow(depth, pose, K, Kinv)
    wt2 = wts(p2f.shape, 2)
    gd, gp = torch.autograd.grad((p2f * wt2).sum(), [depth, pose])
    d.update(p2f_out=p2f, p2f_wt=wt2, p2f_gdepth=gd, p2f_gpose=gp)
    d['p2f_zeros_out'] = RW.pose2flow(depth, pose, K, Kinv, padding_mode='zeros')
    d['posemat_euler'] = RW.pose_vec2mat(pose, 'euler')
    d['posemat_quat'] = RW.pose_vec2mat(pose, 'quat')
    d['oob'] = RW.flow2oob(flow * 4).to(torch.uint8)
    a, b_ = s['tgt'], leaf(fw.detach())
    sm = RS.ssim(a, b_)
    wt3 = wts(sm.shape, 3)
    d.update(ssim_out=sm, ssim_wt=wt3, ssim_gimg2=torch.autograd.grad((sm * wt3).sum(), [b_])[0])
    d.update(img=img, tgt=s['tgt'], depth=depth, pose=pose, K=K, Kinv=Kinv, flow=flow)
    save('warp_small', d)


# --------------------------------------------------------------------------- B. cfg0
def gen_cfg0():
    """BASELINE.json configs[0]: inverse_warp + L1 photometric on one 3x128x416 triplet."""
    B, H, W = 1, 128, 416
    tgt, refs = synth.frames(B, H, W, seed=20, n_refs=2)
    K, Kinv = synth.intrinsics(B, H, W)
    depth = leaf(synth.depths(B, H, W, 1, seed=21)[0][:, 0])
    pose = leaf(synth.poses(B, 2, seed=22, big_tx_sample=False))
    loss = 0
    for i in range(2):
        w = RW.inverse_warp(refs[i], depth, pose[:, i], K, Kinv)
        valid = 1 - (w == 0).prod(1, keepdim=True).type_as(w)
        loss = loss + ((tgt - w) * valid).abs().mean()
    gd, gp = torch.autograd.grad(loss, [depth, pose])
    save('cfg0', dict(loss=loss, gdepth=gd, gpose=gp, B=B, H=H, W=W))


# --------------------------------------------------------------------------- C. loss layer
def gen_losses():
    B, H, W, NL = 2, 64, 96, 3
    s = synth.sample(B, H, W, seed=30, nlevels=NL)
    tgt, refs, K, Kinv = s['tgt'], s['refs'], s['K'], s['Kinv']
    d = dict(B=B, H=H, W=W, NL=NL)
    for tag, wssim in (('w997', 0.997), ('w0', 0.0)):
        for mtag in ('mask', 'nomask'):
            depth = [leaf(x) for x in s['depth']]
            pose = leaf(s['pose'])
            em = [leaf(x) for x in s['emask']] if mtag == 'mask' else [None] * NL
            l = RL.photometric_reconstruction_loss(tgt, refs, K, Kinv, depth, em, pose, wssim=wssim,
                                                   lambda_oob=0.1 if tag == 'w0' else 0)
            ins = depth + [pose] + (em if mtag == 'mask' else [])
            g = torch.autograd.grad(l, ins)
            key = f'rigid_{tag}_{mtag}'
            d[key] = l
            for i in range(NL):
                d[f'{key}_gdepth{i}'] = g[i]
            d[f'{key}_gpose'] = g[NL]
            if mtag == 'mask':
                for i in range(NL):
                    d[f'{key}_gmask{i}'] = g[NL + 1 + i]
        ff = [leaf(x) for x in s['flow_fwd']]
        fb = [leaf(x) for x in s['flow_bwd']]
        em = [leaf(x) for x in s['emask']]
        fem = [1 - m[:, 1:3] for m in em]
        l = RL.photometric_flow_loss(tgt, refs[1:3], [fb, ff], fem, wssim=wssim)
        g = torch.autograd.grad(l, ff + fb + em)
        key = f'flow_{tag}'
        d[key] = l
        for i in range(NL):
            d[f'{key}_gff{i}'], d[f'{key}_gfb{i}'], d[f'{key}_gmask{i}'] = g[i], g[NL + i], g[2 * NL + i]
    # occlusion masks
    d['depth_occ0'] = RL.depth_occlusion_masks(s['depth'][0], s['pose'], K, Kinv)
    d['depth_occ1'] = RL.depth_occlusion_masks(s['depth'][1], s['pose'], K, Kinv)
    # smoothness
    for nm, preds in (('depth', s['depth']), ('flow', s['flow_fwd']), ('mask', s['emask'])):
        pl = [leaf(x) for x in preds]
        l = RL.edge_aware_smoothness_loss(tgt, pl)
        g = torch.autograd.grad(l, pl)
        d[f'edge_{nm}'] = l
        for i in range(NL):
            d[f'edge_{nm}_g{i}'] = g[i]
        pl = [leaf(x) for x in preds]
        l = RL.smooth_loss(pl)
        g = torch.autograd.grad(l, pl)
        d[f'smooth_{nm}'] = l
        for i in range(NL):
            d[f'smooth_{nm}_g{i}'] = g[i]
    # explainability + consensus
    em = [leaf(x) for x in s['emask']]
    l = RL.explainability_loss(em)
    g = torch.autograd.grad(l, em)
    d['expl'] = l
    for i in range(NL):
        d[f'expl_g{i}'] = g[i]
    depth = s['depth']
    cam_f = [RW.pose2flow(x.squeeze(1), s['pose'][:, 2], K, Kinv) for x in depth]
    cam_b = [RW.pose2flow(x.squeeze(1), s['pose'][:, 1], K, Kinv) for x in depth]
    # make the flows partly agree with the rigid flow so both target classes occur
    ff = [0.5 * a + 0.5 * b for a, b in zip(cam_f, s['flow_fwd'])]
    fb = [0.5 * a + 0.5 * b for a, b in zip(cam_b, s['flow_bwd'])]
    for i in range(NL):
        d[f'cons_ff{i}'], d[f'cons_fb{i}'] = ff[i], fb[i]
    tg = RL.consensus_exp_masks(cam_f, cam_b, ff, fb, tgt, refs[2], refs[1], wssim=0.997, wrig=1.0, ws=0.1)
    for i in range(NL):
        d[f'cons_target{i}'] = tg[i]
        d[f'cam_f{i}'], d[f'cam_b{i}'] = cam_f[i], cam_b[i]
    rig_f = [(a - b).abs() for a, b in zip(cam_f, ff)]
    rig_b = [(a - b).abs() for a, b in zip(cam_b, fb)]
    em = [leaf(x) for x in s['emask']]
    l = RL.consensus_depth_flow_mask(em, rig_b, rig_f, tg, tg, THRESH=0.5, wbce=0.3)
    g = torch.autograd.grad(l, em)
    d['cdfm'] = l
    for i in range(NL):
        d[f'cdfm_g{i}'] = g[i]
    save('loss_small', d)


# --------------------------------------------------------------------------- D. nets
def load_ref(mod, params):
    sd = {k: v.clone() for k, v in params.items()}
    missing = mod.load_state_dict(sd, strict=True)
    return mod


def gen_nets():
    d = {}
    B, H, W = 2, 64, 128         # DispResNet6 / PoseNetB6 (smaller inputs make the deepest BatchNorms, which see
                                 # only B*1*1 values, ill-conditioned: fp32 summation order then changes grads by %)
    tgt, refs = synth.frames(B, H, W, seed=40)
    # DispResNet6
    P = onets.disp_params()
    net = load_ref(RM.DispResNet6(), P)
    net.train()
    disps = net(tgt)
    wt = [wts(x.shape, 50 + i) for i, x in enumerate(disps)]
    loss = sum((x * w_).sum() for x, w_ in zip(disps, wt))
    names = ['conv1.0.weight', 'conv1.2.bias', 'conv2.0.conv1.weight', 'conv2.0.downsample.0.weight',
             'conv2.0.downsample.1.weight', 'conv2.0.downsample.1.bias', 'conv7.1.conv2.weight',
             'upconv7.0.weight', 'upconv1.0.bias', 'iconv1.0.conv1.weight', 'iconv3.0.downsample.0.weight',
             'predict_disp1.0.weight', 'predict_disp6.0.bias']
    pd = dict(net.named_parameters())
    g = torch.autograd.grad(loss, [pd[n] for n in names])
    for i, x in enumerate(disps):
        d[f'disp_out{i}'] = x
    for n, gg in zip(names, g):
        sfx, gg = compact(gg)
        d['disp_g_' + n + sfx] = gg
    sd = net.state_dict()
    d['disp_rm'] = sd['conv2.0.downsample.1.running_mean'].clone()
    d['disp_rv'] = sd['iconv1.0.downsample.1.running_var'].clone()
    net.eval()
    d['disp_eval'] = net(tgt)
    # odd size: crop_like path (128x416-like aspect: 40x104)
    t2, _ = synth.frames(2, 24, 40, seed=41)
    net.train()
    o2 = net(t2)
    for i, x in enumerate(o2):
        d[f'disp_odd_out{i}'] = x
    # PoseNetB6
    Pp = onets.pose_params()
    pnet = load_ref(RM.PoseNetB6(nb_ref_imgs=4), Pp)
    pose = pnet(tgt, refs)
    wtp = wts(pose.shape, 60)
    ppd = dict(pnet.named_parameters())
    pn = ['conv1.0.weight', 'conv2.0.weight', 'conv8.0.bias', 'pose_pred.weight', 'pose_pred.bias']
    g = torch.autograd.grad((pose * wtp).sum(), [ppd[n] for n in pn])
    d['pose_out'] = pose
    for n, gg in zip(pn, g):
        sfx, gg = compact(gg)
        d['pose_g_' + n + sfx] = gg
    # MaskNet6 / Back2Future need H, W divisible by 64 (SURVEY F8)
    B, H, W = 1, 64, 64
    tgt, refs = synth.frames(B, H, W, seed=42)
    Pm = onets.mask_params()
    mnet = load_ref(RM.MaskNet6(nb_ref_imgs=4, output_exp=True), Pm)
    mnet.train()
    ms = mnet(tgt, refs)
    wm = [wts(x.shape, 70 + i) for i, x in enumerate(ms)]
    mpd = dict(mnet.named_parameters())
    mn = ['conv1.0.weight', 'conv6.0.weight', 'deconv6.0.weight', 'deconv1.0.weight', 'deconv3.0.bias',
          'pred_mask1.weight', 'pred_mask6.bias']
    g = torch.autograd.grad(sum((x * w_).sum() for x, w_ in zip(ms, wm)), [mpd[n] for n in mn])
    for i, x in enumerate(ms):
        d[f'mask_out{i}'] = x
    for n, gg in zip(mn, g):
        sfx, gg = compact(gg)
        d['mask_g_' + n + sfx] = gg
    # Back2Future (stub correlation)
    Pf = onets.flow_params()
    fnet = load_ref(RM.Back2Future(nlevels=6), Pf)
    fnet.train()
    ff, fb, occ = fnet(tgt, refs[1:3])
    wf = [wts(x.shape, 80 + i) for i, x in enumerate(ff)]
    fpd = dict(fnet.named_parameters())
    fn = ['conv1a.0.weight', 'conv1b.2.bias', 'conv6c.0.weight', 'decoder_fwd6.0.weight',
          'decoder_bwd2.10.weight', 'decoder_fwd2.0.weight', 'decoder_bwd4.4.bias']
    g = torch.autograd.grad(sum((x * w_).sum() + (y * w_).sum() * 0.5 for x, y, w_ in zip(ff, fb, wf)),
                            [fpd[n] for n in fn])
    for i in range(6):
        d[f'flow_fwd{i}'], d[f'flow_bwd{i}'] = ff[i], fb[i]
    d['flow_occ0'], d['flow_occ5'] = occ[0][:, :, ::4, ::4], occ[5]
    for n, gg in zip(fn, g):
        sfx, gg = compact(gg)
        d['flow_g_' + n + sfx] = gg
    fnet.eval()
    e = fnet(tgt, refs[1:3])
    d['flow_eval_fwd'] = e[0][:, :, ::2, ::2]
    save('nets_small', d)
    return dict(disp=net, pose=pnet, mask=mnet, flow=fnet)


# --------------------------------------------------------------------------- E. full step body
def gen_step(nets_):
    """Reference train.py:454-509 executed verbatim on reference modules/functions, B=2 64x128."""
    B, H, W = 2, 64, 128
    tgt, refs = synth.frames(B, H, W, seed=40)
    K, Kinv = synth.intrinsics(B, H, W)
    disp_net, pose_net, mask_net, flow_net = [nets_[k] for k in ('disp', 'pose', 'mask', 'flow')]
    for n, P in zip((disp_net, pose_net, mask_net, flow_net),
                    (onets.disp_params(), onets.pose_params(), onets.mask_params(), onets.flow_params())):
        load_ref(n, P)
        n.train()
        n.zero_grad()
    w1, w2, w3, w4, w5 = 1.0, 0.1, 0.1, 0.5, 0.3
    wssim, THRESH, wbce, wrig = 0.997, 0.01, 0.5, 1.0
    disparities = disp_net(tgt)
    depth = [1 / disp for disp in disparities]
    pose = pose_net(tgt, refs)
    explainability_mask = mask_net(tgt, refs)
    flow_fwd, flow_bwd, _ = flow_net(tgt, refs[1:3])
    flows_cam_fwd = [RW.pose2flow(d_.squeeze(1), pose[:, 2], K, Kinv) for d_ in depth]
    flows_cam_bwd = [RW.pose2flow(d_.squeeze(1), pose[:, 1], K, Kinv) for d_ in depth]
    exp_masks_target = RL.consensus_exp_masks(flows_cam_fwd, flows_cam_bwd, flow_fwd, flow_bwd, tgt, refs[2],
                                              refs[1], wssim=wssim, wrig=wrig, ws=w3)
    rigidity_mask_fwd = [(a - b).abs() for a, b in zip(flows_cam_fwd, flow_fwd)]
    rigidity_mask_bwd = [(a - b).abs() for a, b in zip(flows_cam_bwd, flow_bwd)]
    flow_exp_mask = [1 - m[:, 1:3] for m in explainability_mask]
    loss_1 = RL.photometric_reconstruction_loss(tgt, refs, K, Kinv, depth, explainability_mask, pose,
                                                lambda_oob=0, qch=0.5, wssim=wssim)
    loss_2 = RL.explainability_loss(explainability_mask)
    loss_3 = RL.edge_aware_smoothness_loss(tgt, depth) + RL.edge_aware_smoothness_loss(tgt, flow_fwd)
    loss_3 = loss_3 + RL.edge_aware_smoothness_loss(tgt, flow_bwd) + RL.edge_aware_smoothness_loss(tgt, explainability_mask)
    loss_4 = RL.photometric_flow_loss(tgt, refs[1:3], [flow_bwd, flow_fwd], flow_exp_mask, lambda_oob=0,
                                      qch=0.5, wssim=wssim)
    loss_5 = RL.consensus_depth_flow_mask(explainability_mask, rigidity_mask_bwd, rigidity_mask_fwd,
                                          exp_masks_target, exp_masks_target, THRESH=THRESH, wbce=wbce)
    loss = w1 * loss_1 + w2 * loss_2 + w3 * loss_3 + w4 * loss_4 + w5 * loss_5
    loss.backward()
    d = dict(loss=loss, loss_1=loss_1, loss_2=loss_2, loss_3=loss_3, loss_4=loss_4, loss_5=loss_5)
    pick = dict(disp=['conv1.0.weight', 'predict_disp1.0.weight', 'iconv4.0.conv2.weight'],
                pose=['conv1.0.weight', 'pose_pred.bias'],
                mask=['conv1.0.weight', 'pred_mask1.weight'],
                flow=['conv1a.0.weight', 'decoder_fwd2.10.weight'])
    for nm, net in (('disp', disp_net), ('pose', pose_net), ('mask', mask_net), ('flow', flow_net)):
        pd = dict(net.named_parameters())
        gn = torch.sqrt(sum((p.grad ** 2).sum() for p in pd.values() if p.grad is not None))
        d[f'gnorm_{nm}'] = gn
        for n in pick[nm]:
            sfx, gg = compact(pd[n].grad)
            d[f'g_{nm}_{n}{sfx}'] = gg
    # cfg1 composition (mask None) on the same nets
    for n in (disp_net, pose_net):
        n.zero_grad()
    disparities = disp_net(tgt)
    depth = [1 / disp for disp in disparities]
    pose = pose_net(tgt, refs)
    l1 = RL.photometric_reconstruction_loss(tgt, refs, K, Kinv, depth, [None] * 6, pose, wssim=wssim)
    l3 = RL.edge_aware_smoothness_loss(tgt, depth)
    (w1 * l1 + w3 * l3).backward()
    d['cfg1_loss'], d['cfg1_l1'], d['cfg1_l3'] = w1 * l1 + w3 * l3, l1, l3
    pd = dict(disp_net.named_parameters())
    d['cfg1_g_disp_conv1.0.weight'] = pd['conv1.0.weight'].grad
    d['cfg1_gnorm_disp'] = torch.sqrt(sum((p.grad ** 2).sum() for p in pd.values()))
    pd = dict(pose_net.named_parameters())
    d['cfg1_g_pose_pose_pred.bias'] = pd['pose_pred.bias'].grad
    save('step_small', d)


# --------------------------------------------------------------------------- F. validation metrics (N2)
def gen_metrics():
    """Reference loss_functions.py:355-467 on synthetic KITTI-like ground truth (sparse valid mask, odd sizes)."""
    g = torch.Generator().manual_seed(70)
    B, Hg, Wg, hp, wp, hm, wm = 2, 37, 122, 16, 52, 8, 26
    gt = torch.cat((torch.randn(B, 2, Hg, Wg, generator=g) * 6, (torch.rand(B, 1, Hg, Wg, generator=g) > 0.6).float()), 1)
    pr, pn = torch.randn(B, 2, hp, wp, generator=g) * 2, torch.randn(B, 2, hp, wp, generator=g) * 2
    mask = torch.rand(B, 1, hm, wm, generator=g)
    d = dict(gt=gt, pr=pr, pn=pn, mask=mask)
    d['flow_diff'] = RL.flow_diff(gt, pr)
    d['epe3'] = torch.tensor(RL.compute_epe(gt, pr))
    d['epe2'] = torch.tensor(RL.compute_epe(gt[:, :2].contiguous(), pr))
    d['outlier'] = torch.tensor(RL.outlier_err(gt, pr * 3))
    d['all_epes'] = torch.tensor(RL.compute_all_epes(gt, pr, pn, mask))
    d['all_epes_t3'] = torch.tensor(RL.compute_all_epes(gt, pr, pn, mask, THRESH=0.3))
    Bd, H, W = 3, 48, 160
    dgt = torch.rand(Bd, H, W, generator=g) * 100 - 10          # some <= 0 and >= 80: invalid
    dpr = torch.rand(Bd, H, W, generator=g) * 60 + 0.5
    dpr[0, :5] = 1e-5                                            # clamp path
    d.update(dgt=dgt, dpr=dpr)
    d['errors_crop'] = torch.stack([torch.as_tensor(v) for v in RL.compute_errors(dgt, dpr, crop=True)])
    d['errors_nocrop'] = torch.stack([torch.as_tensor(v) for v in RL.compute_errors(dgt, dpr, crop=False)])
    save('metrics_small', d)


# --------------------------------------------------------------------------- G. input transforms (N1)
def gen_transforms():
    """The reference's train transform (custom_transforms.py, train.py:165-172) on uint8 frames.  scipy.misc (removed from
    scipy) is stubbed with its historical implementation: imresize(arr, size) = PIL resize with BILINEAR (scipy 1.1
    misc/pilutil.py)."""
    import random as pyrandom
    from PIL import Image
    misc = types.ModuleType('scipy.misc')
    misc.imresize = lambda arr, size: np.array(Image.fromarray(arr).resize((size[1], size[0]), resample=Image.BILINEAR))
    misc.imrotate = lambda arr, angle: arr
    sys.modules['scipy.misc'] = misc
    import scipy
    scipy.misc = misc
    import custom_transforms as CT
    rs = np.random.RandomState(5)
    B, F, Hs, Ws = 3, 5, 32, 48
    frames = rs.randint(0, 256, size=(B, F, Hs, Ws, 3)).astype(np.uint8)
    K = np.array([[30.5, 0, 24.2], [0, 31.5, 15.1], [0, 0, 1]], np.float32)
    tf = CT.Compose([CT.RandomHorizontalFlip(), CT.RandomScaleCrop(), CT.ArrayToTensor(), CT.Normalize(mean=[0.5, 0.5, 0.5], std=[0.5, 0.5, 0.5])])
    pyrandom.seed(11)
    np.random.seed(12)
    outs, Ks = [], []
    for b in range(B):
        imgs, Kb = tf([frames[b, f] for f in range(F)], np.copy(K))
        outs.append(torch.stack(imgs))
        Ks.append(torch.from_numpy(np.asarray(Kb, np.float32)))
    d = dict(frames=frames, K=K, out=torch.stack(outs), K_out=torch.stack(Ks), seed_random=11, seed_np=12)
    # no-resize variant (flip + normalise only): must be reproduced exactly
    tf2 = CT.Compose([CT.RandomHorizontalFlip(), CT.ArrayToTensor(), CT.Normalize(mean=[0.5, 0.5, 0.5], std=[0.5, 0.5, 0.5])])
    pyrandom.seed(13)
    outs2, K2 = [], []
    for b in range(B):
        imgs, Kb = tf2([frames[b, f] for f in range(F)], np.copy(K))
        outs2.append(torch.stack(imgs))
        K2.append(torch.from_numpy(np.asarray(Kb, np.float32)))
    d.update(out_flip=torch.stack(outs2), K_flip=torch.stack(K2), seed_flip=13)
    save('transforms_small', d)


# --------------------------------------------------------------------------- H. helper exports (a17) + B2F tables
def gen_helpers():
    """The small functions the reference module exports next to the losses (loss_functions.py:13-25,132-158,204-219,
    252-261,343-352) and the channel-permutation tables Back2Future builds (models/back2future.py:56-59)."""
    B, H, W, NL = 2, 32, 48, 3
    s = synth.sample(B, H, W, seed=33, nlevels=NL)
    d = dict(B=B, H=H, W=W, NL=NL)
    d['spatial_normalize'] = RL.spatial_normalize(s['depth'][0])
    x = s['flow_fwd'][0]
    d['robust_l1'] = RL.robust_l1(x)
    d['robust_l1_q'] = RL.robust_l1(x, q=0.35, eps=1e-3)
    d['robust_l1_per_pix'] = RL.robust_l1_per_pix(x)
    ob, of = RL.occlusion_masks(s['flow_bwd'][0] * 3, s['flow_fwd'][0] * 3)
    d['occ_bw'], d['occ_fw'] = ob, of
    d['depth_occ'] = RL.depth_occlusion_masks(s['depth'][0], s['pose'], s['K'], s['Kinv'])
    d['gauss_expl'] = RL.gaussian_explainability_loss(s['emask'])
    d['logical_or'] = RL.logical_or(s['emask'][0][:, :2], s['emask'][0][:, 2:])
    rig_f = [(a - b).abs() for a, b in zip(s['flow_fwd'], s['flow_bwd'])]
    rig_b = [(a + b).abs() * 0.5 for a, b in zip(s['flow_fwd'], s['flow_bwd'])]
    jm = RL.compute_joint_mask_for_depth(s['emask'], rig_b, rig_f, 0.5)
    for i in range(NL):
        d[f'joint{i}'] = jm[i]
    tgt = (s['emask'][0] > 0.5).float()
    d['wbce'] = RL.weighted_binary_cross_entropy(s['emask'][0], tgt, [0.3, 0.7])
    d['wbce_none'] = RL.weighted_binary_cross_entropy(s['emask'][0], tgt)
    m = RM.Back2Future(nlevels=6)
    d['idx_fwd'], d['idx_bwd'] = m.idx_fwd.cpu(), m.idx_bwd.cpu()
    save('helpers_small', d)


# --------------------------------------------------------------------------- I. alternate nets (SURVEY N4)
ALT_NETS = [  # name, constructor kwargs, input size (B, H, W), parameters whose gradients are frozen
    ('DispNetS', {}, (2, 64, 128), ['conv1.0.weight', 'conv7.2.bias', 'upconv4.0.weight', 'iconv3.0.weight', 'predict_disp4.0.weight']),
    ('DispNetS6', {}, (2, 64, 128), ['conv1.2.weight', 'conv5.0.bias', 'upconv7.0.weight', 'iconv1.0.weight', 'predict_disp6.0.bias']),
    ('DispResNetS6', {}, (2, 64, 128), ['conv1.0.weight', 'conv4.2.conv2.weight', 'iconv5.1.conv1.weight', 'iconv7.0.downsample.1.bias',
                                       'predict_disp1.0.weight']),
    ('PoseNet6', dict(nb_ref_imgs=4), (2, 128, 128), ['conv0.0.weight', 'conv1.0.weight', 'conv7.0.bias', 'pose_pred.weight']),
    ('PoseExpNet', dict(nb_ref_imgs=4, output_exp=True), (2, 64, 128), ['conv1.0.weight', 'conv6.0.weight', 'upconv5.0.weight',
                                                                      'upconv1.0.bias', 'predict_mask4.weight', 'pose_pred.bias']),
    ('MaskResNet6', dict(nb_ref_imgs=4, output_exp=True), (2, 128, 128), ['conv1.0.weight', 'conv3.0.downsample.1.weight', 'conv6.1.conv2.weight',
                                                                        'deconv6.0.weight', 'deconv1.0.bias', 'pred_mask1.weight']),
]


def alt_outputs(name, net, tgt, refs):
    """The tensors of one alternate net that the fixture holds (train mode)."""
    if name.startswith('Disp'):
        return list(net(tgt))
    if name == 'PoseNet6':
        return [net(tgt, refs)]
    if name == 'PoseExpNet':
        masks, pose = net(tgt, refs)
        return list(masks) + [pose]
    return list(net(tgt, refs))


def gen_alt_nets():
    d = {}
    for k, (name, kw, (B, H, W), pn) in enumerate(ALT_NETS):
        tgt, refs = synth.frames(B, H, W, seed=190 + k)
        net = synth.seeded_fill(getattr(RM, name)(**kw), 300 + k)
        net.train()
        outs = alt_outputs(name, net, tgt, refs)
        loss = sum((x * wts(x.shape, 400 + 10 * k + i)).sum() for i, x in enumerate(outs))
        pd = dict(net.named_parameters())
        g = torch.autograd.grad(loss, [pd[n] for n in pn])
        for i, x in enumerate(outs):
            d[f'{name}_out{i}'] = x
        for n, gg in zip(pn, g):
            sfx, gg = compact(gg)
            d[f'{name}_g_{n}{sfx}'] = gg
        net.eval()
        e = net(tgt) if name.startswith('Disp') else net(tgt, refs)
        d[f'{name}_eval'] = e if torch.is_tensor(e) else (e[1] if name == 'PoseExpNet' else e[0])
    save('alt_nets_small', d)


if __name__ == '__main__':
    if 'alt' in sys.argv:                  # only the alternate-net fixture
        gen_alt_nets()
        sys.exit(0)
    if 'extra' in sys.argv:                # only the round-2 fixtures (the round-1 files stay byte-identical)
        gen_metrics()
        gen_transforms()
        gen_helpers()
        sys.exit(0)
    gen_warp()
    gen_cfg0()
    gen_losses()
    ns = gen_nets()
    gen_step(ns)
    gen_metrics()
    gen_transforms()
    gen_helpers()
