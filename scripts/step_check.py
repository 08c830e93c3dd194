"""Staged hardware checks of the coupling-step kernel (nfk_rq_coupling_step_f16x3), smallest configuration first.
usage: step_check.py <stage>     (each stage is run in its own process by scripts/step_check.sh, under `timeout`)"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nflows_b200 import _native as N
from nflows_b200 import dense as D
from nflows_b200 import kernels as K
from nflows_b200.nn.nets import ResidualNet

dev = torch.device("cuda:0")


def rel(a, b):
    a, b = a.double(), b.double()
    return float(((a - b).abs() / torch.maximum(torch.maximum(a.abs(), b.abs()), torch.ones_like(a))).max())


def trunk(hidden, blocks, rows, in_features, scale=0.05):
    torch.manual_seed(hidden + blocks + in_features)
    net = ResidualNet(in_features, 16, hidden_features=hidden, num_blocks=blocks).eval()
    with torch.no_grad():
        for p in net.parameters():
            p.add_(torch.randn_like(p) * scale)
        x = torch.randn(rows, in_features)
        h = net.double().initial_layer(x.double())
        for block in net.blocks:
            h = block(h)
        net = net.float().to(dev)
        chain = net.dense_chain(None)
        flags = K.new_flags(dev)
        xp = K.split_f16(x.to(dev), D.act_exp(), flags=flags)
        plan = D.step_plan(chain)
        out = K.Pair16.empty(rows, hidden, D.act_exp(), dev)
        out.hi.fill_(float("nan")); out.lo.fill_(float("nan"))
        K.rq_coupling_step(plan, xp, h_pair=out, flags=flags)
        torch.cuda.synchronize()
        got = out.float().cpu()
        base = D.run_trunk(chain, x.to(dev), None, True).pair.float().cpu()
    print("trunk H=%d blocks=%d rows=%d K0=%d flags=%s: step vs fp64 %.2e, r1 path vs fp64 %.2e, step vs r1 %.2e, device flags %d" % (
        hidden, blocks, rows, in_features, plan.layer_flags, rel(got, h), rel(base, h), rel(got, base), int(flags.item())))
    bad = (got - h.float()).abs().max(dim=1).values
    if rel(got, h) > 1e-5:
        idx = torch.nonzero(bad > 1e-4).flatten()
        print("   bad rows: %d of %d, first %s" % (idx.numel(), rows, idx[:16].tolist()))
        badc = (got - h.float()).abs().max(dim=0).values
        idc = torch.nonzero(badc > 1e-4).flatten()
        print("   bad cols: %d of %d, first %s" % (idc.numel(), hidden, idc[:32].tolist()))


def coupling(features, hidden, blocks, rows, bins=8, tails="linear", inverse=False, final_scale=3.0):
    from nflows_b200 import config, transforms as T
    from nflows_b200.utils import torchutils
    torch.manual_seed(features + hidden + bins)
    t = T.PiecewiseRationalQuadraticCouplingTransform(
        mask=torchutils.create_alternating_binary_mask(features),
        transform_net_create_fn=lambda i, o: ResidualNet(i, o, hidden_features=hidden, num_blocks=blocks),
        num_bins=bins, tails=tails, tail_bound=3.0 if tails else 1.0).eval()
    with torch.no_grad():
        t.transform_net.final_layer.weight.mul_(final_scale)
        t.transform_net.final_layer.bias.mul_(final_scale)
        x = torch.randn(rows, features) if tails else torch.rand(rows, features)
        want_y, want_l = (t.double().inverse if inverse else t.double().forward)(x.double())
        t = t.float().to(dev)
        fn = t.inverse if inverse else t.forward
        config.coupling_step_kernel = True
        c0 = N.launch_count()
        y, l = fn(x.to(dev))
        torch.cuda.synchronize()
        launches = N.launch_count() - c0
        config.coupling_step_kernel = False
        y0, l0 = fn(x.to(dev))
        torch.cuda.synchronize()
        config.coupling_step_kernel = True
    print("coupling D=%d H=%d blocks=%d rows=%d K=%d tails=%s inv=%d: step y %.2e lad %.2e | r1 path y %.2e lad %.2e | step vs r1 y %.2e lad %.2e | %d launches" % (
        features, hidden, blocks, rows, bins, tails, inverse, rel(y.cpu(), want_y), rel(l.cpu(), want_l), rel(y0.cpu(), want_y),
        rel(l0.cpu(), want_l), rel(y.cpu(), y0.cpu()), rel(l.cpu(), l0.cpu()), launches))
    if rel(y.cpu(), want_y) > 1e-4:
        bad = (y.cpu() - want_y.float()).abs()
        rows_bad = torch.nonzero(bad.max(dim=1).values > 1e-3).flatten()
        cols_bad = torch.nonzero(bad.max(dim=0).values > 1e-3).flatten()
        print("   bad rows %d (first %s) bad cols %d (first %s)" % (rows_bad.numel(), rows_bad[:12].tolist(), cols_bad.numel(), cols_bad[:24].tolist()))
        idx = torch.nonzero(bad > 1e-3)
        tf = t.transform_features.cpu().tolist()
        for r_, c_ in idx[:24].tolist():
            j = tf.index(c_) if c_ in tf else -1
            print("      row %d (tile %d, r %d) col %d (feature %d: tile n=%d, slot %d) got %.5f want %.5f x %.5f r1path %.5f" % (
                r_, r_ // 128, r_ % 128, c_, j, j // 8, j % 8, float(y[r_, c_]), float(want_y[r_, c_]), float(x[r_, c_]), float(y0[r_, c_])))
        tiles = sorted(set((r_ // 128) for r_, _ in idx.tolist()))
        print("      tiles with errors:", tiles[:40], "features:", sorted(set(tf.index(c_) for _, c_ in idx.tolist() if c_ in tf))[:40])


STAGES = {
    "t0": lambda: trunk(64, 0, 128, 40),          # initial layer only, one tile
    "t1": lambda: trunk(64, 1, 130, 40),          # one residual block, two tiles
    "t2": lambda: trunk(256, 2, 1000, 40),        # cfg-3 widths
    "t3": lambda: trunk(128, 3, 4096, 392),       # long initial layer (13 K-slabs: wraps the 4-stage ring), 6 square layers
    "t4": lambda: trunk(256, 2, 40000, 392),      # more tiles than CTAs: the persistent loop, ring reuse across tiles
    "c0": lambda: coupling(16, 64, 1, 128),
    "c1": lambda: coupling(64, 128, 2, 5000),
    "c2": lambda: coupling(64, 128, 2, 5000, inverse=True),
    "c3": lambda: coupling(784, 256, 2, 20000),
    "c4": lambda: coupling(48, 96, 2, 3000, bins=10),
    "c5": lambda: coupling(48, 64, 1, 3000, bins=4),
    "c6": lambda: coupling(48, 64, 1, 3000, bins=16),
    "c7": lambda: coupling(48, 64, 1, 3000, bins=8, tails=None),
    "c8": lambda: coupling(48, 64, 1, 3000, bins=16, tails=None, inverse=True),
}

if __name__ == "__main__":
    STAGES[sys.argv[1]]()
