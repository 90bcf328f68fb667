"""Development aid: determinism and accuracy of the pooled eigen-solver (cluster Jacobi) on repeated launches."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import vit_bias_aware_structural_distillation_b200 as pkg
lib = pkg.load(); dev = torch.device("cuda:0")
st = torch.cuda.current_stream().cuda_stream
for n in (36, 50, 64, 100, 192):
    torch.manual_seed(n)
    X = torch.randn(4 * n, n) * (0.97 ** torch.arange(n))
    G = (X.T @ X).to(dev)
    outs = []
    for rep in range(12):
        ev = torch.zeros(n, device=dev); evec = torch.zeros(n, n, device=dev)
        sw = torch.zeros(4, dtype=torch.int32, device=dev)
        ws = torch.zeros(4 * (2 * n * n + n) + 8192, dtype=torch.uint8, device=dev)
        rc = lib.basd_selftest_eig(G.data_ptr(), n, ev.data_ptr(), evec.data_ptr(), sw.data_ptr(), ws.data_ptr(), st)
        assert rc == 0
        torch.cuda.synchronize()
        outs.append((ev.cpu(), evec.cpu(), sw[0].item()))
    same = all(torch.equal(outs[0][0], o[0]) and torch.equal(outs[0][1], o[1]) for o in outs)
    ref = torch.linalg.eigvalsh(G.cpu().double()).flip(0)
    V = outs[0][1].double()
    print(f"n={n}: bitwise identical over 12 launches: {same}; sweeps {sorted(set(o[2] for o in outs))}; "
          f"eval err {((outs[0][0].double() - ref).abs().max() / ref.max()).item():.2e}; "
          f"orth {(V @ V.T - torch.eye(n, dtype=torch.float64)).abs().max().item():.2e}")

