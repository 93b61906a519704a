"""Per-kernel timing of the hot path at a given size (developer tool)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import seam_match_rcnn_b200 as pkg
from bench import random_init_weights
dev = torch.device("cuda:0")
e = pkg.SeamEngine(dev); e.load_weights(random_init_weights(dev))
Q, T, G = [int(x) for x in (sys.argv[1:4] if len(sys.argv) > 3 else (15000, 10, 15000))]
seq = torch.randn(1 + T, Q, 256, device=dev)
q = e.aggregate(seq)
gal = e.prepare_gallery(torch.randn(G, 256, device=dev)) if G else None
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
for it in range(3):
    e.aggregate(seq)
    if G: e.score_topk(q, gal, 20)
e.profile(True)
for it in range(10):
    flush.fill_(1)
    e.aggregate(seq)
    if G: e.score_topk(q, gal, 20)
torch.cuda.synchronize()
pr = e.profile_read()
extra = ""
if G:
    plan = e.score_plan(Q, G)
    ws = e._ws["score"]
    nl = plan["ctas_per_query_tile"] * 4
    cn = ws[plan["off_rowcnt"]:plan["off_rowcnt"] + Q * nl * 4].view(torch.int32).view(Q, nl).float()
    _, _, _, st = e.score_topk(q, gal, 20, return_stats=True)
    extra = (f" | P={plan['ctas_per_query_tile']} cap={plan['list_capacity']} sublist max={int(cn.max())} "
             f"row total mean={cn.sum(1).mean():.0f} max={int(cn.sum(1).max())} fallback_rows={int(st[0])} "
             f"ws={plan['bytes'] / 2**20:.0f} MiB")
print(f"Q={Q} T={T} G={G}: " + ", ".join(f"{k}={v[0]/v[1]*1e3:.1f}us" for k, v in pr.items() if v[1]) + extra)
