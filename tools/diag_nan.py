"""diagnostic: first non-finite tensor in a C5-shaped training run (B 2048, 20000 genes)"""
import sys
import torch
sys.path.insert(0, ".")
from spvipes_b200 import synth
from spvipes_b200.engine import GroupBatch, StepEngine
from spvipes_b200.trainer import TrainLoop, init_params

B, G, H, N = 2048, 20000, 128, 16384
prec = sys.argv[1] if len(sys.argv) > 1 else "bf16"
data = synth.make_counts((N, N), (G, G), 10, device="cuda", seed=1234)
eng = StepEngine((G, G), H, 25, 10, 0.1, "label", "cuda", seed=0, precision=prec)
init_params(eng, 0)
loop = TrainLoop(eng)
loop.set_epoch(1)
gen = torch.Generator(device="cuda").manual_seed(5)
for s in range(30):
    rows = [torch.randperm(N, generator=gen, device="cuda")[:B].to(torch.int32) for _ in (0, 1)]
    bt = [GroupBatch(X=data.X[g], rows=rows[g], labels=data.labels[g], labels_per_cell=True) for g in (0, 1)]
    loop.step(bt)
    torch.cuda.synchronize()
    ws = eng._ctx["ws"]
    bad = []
    for g, w in enumerate(ws):
        for k, v in vars(w).items():
            if torch.is_tensor(v) and v.is_floating_point() and k not in ("ws", "ws2", "ws3", "part_nb", "part_stats", "pi", "dyp", "dys", "dpi", "colpart"):
                if not bool(torch.isfinite(v.float()).all()):
                    bad.append((g, k, int((~torch.isfinite(v.float())).sum())))
    fin = bool(torch.isfinite(eng.grads).all()) and bool(torch.isfinite(eng.params.flat).all())
    print(s, "loss", [round(float(x), 3) for x in eng.loss_out[:7]], "grads/params finite", fin, "bad", bad[:12], flush=True)
    if bad or not fin:
        for g, w in enumerate(ws):
            print(" g", g, "max |E4T|", float(w.E4T.float().abs().max()), "max |amixb|", float(w.amixb.float().abs().max()), "max |wzf|", float(w.wzf.float().abs().max()),
                  "max |Wstack|", float(w.Wstack.float().abs().max()), "max |zcb|", float(w.zcb.float().abs().max()), "max lib", float(w.lib.max()), "max rowc", w.rowc.abs().max(0).values.tolist())
        break
