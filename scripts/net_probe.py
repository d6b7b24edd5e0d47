import os, sys, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import net_ref
from chinesecheckersagent_b200.engine import Engine
from chinesecheckersagent_b200.model import ResidualCNN
G = os.path.join(ROOT, 'tests', 'golden')
gold = np.load(os.path.join(G, 'net_golden.npz'))
m = ResidualCNN(engine=Engine(0)).load_weights(os.path.join(G, 'good_model_weights.npz'))
planes = torch.from_numpy(gold['planes']).cuda()
for k in ('simt', 'tc-bf16', 'tc-fp16'):
    m.set_kernel(k.split('-')[0], tc_dtype=k.split('-')[1] if '-' in k else None)
    l, v = m.forward(planes)
    l = l.cpu().numpy().astype(np.float64); v = v.cpu().numpy().astype(np.float64)
    p_ref = net_ref.softmax64(gold['logits']); p = net_ref.softmax64(l)
    dl = np.abs(l - gold['logits'])
    print(k, 'max|dlogit| %.4g mean %.4g  max|dp| %.4g mean|dp| %.3g  max|dv| %.4g mean %.3g  argmax agree %.4f' % (
        dl.max(), dl.mean(), np.abs(p - p_ref).max(), np.abs(p - p_ref).mean(), np.abs(v - gold['v']).max(), np.abs(v - gold['v']).mean(),
        (p.argmax(1) == p_ref.argmax(1)).mean()))
# timing
big = torch.randint(0, 7, (65536, 7, 7, 7), dtype=torch.uint8, device='cuda')
for k in ('simt', 'tc'):
    m.set_kernel(k)
    m.forward(big); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5): m.forward(big)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 5
    print(k, 'forward 65536 positions: %.3f ms -> %.3g positions/s' % (ms, 65536 / ms * 1e3))
small = big[:4096]
for k in ('simt', 'tc'):
    m.set_kernel(k)
    m.forward(small); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20): m.forward(small)
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 20
    print(k, 'forward 4096 positions: %.3f ms -> %.3g positions/s' % (ms, 4096 / ms * 1e3))
