"""SHA-256 of the raw outputs of the kernels the field-count change touched, at shapes the parent already served, on seeded
inputs -- one line per (entry point, shape, output), so two builds can be compared byte for byte:

    python scratch/fields_bits.py OUT_FILE      (then `cmp` the files of two trees)

Pair dots (rlctr_pairdots_fwd / _bwd, ip_first 0 and 1) at F in {2, 15, 23} and D in {1, 10, 32}; FFM (rlctr_ffm_fwd) logits,
pctr and partner rows at F in {2, 15, 24, 32} and D in {3, 8, 11} (odd D: the per-element partner path)."""
import ctypes as C
import hashlib
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_ctr_prediction_b200 import _lib  # noqa: E402


def digest(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def main(out):
    lib = _lib.load()
    dev = torch.device("cuda:0")
    st = _lib.stream()
    lines = []
    B = 4099
    for F in (2, 15, 23):
        for D in (1, 10, 32):
            g = torch.Generator().manual_seed(F * 1000 + D)
            fd, P = F * D, F * (F - 1) // 2
            rows = torch.randn(B, fd, generator=g).to(dev)
            gout = torch.randn(B, fd + P, generator=g).to(dev)
            for ipf in (0, 1):
                out_ = torch.zeros(B, fd + P, device=dev)
                grows = torch.zeros(B, fd, device=dev)
                _lib.check(lib.rlctr_pairdots_fwd(rows.data_ptr(), fd, out_.data_ptr(), fd + P, B, F, D, ipf, st), "rlctr_pairdots_fwd")
                _lib.check(lib.rlctr_pairdots_bwd(rows.data_ptr(), fd, gout.data_ptr(), fd + P, grows.data_ptr(), fd, B, F, D, ipf, st),
                           "rlctr_pairdots_bwd")
                lines.append(f"pairdots_fwd F={F} D={D} ip_first={ipf} {digest(out_)}")
                lines.append(f"pairdots_bwd F={F} D={D} ip_first={ipf} {digest(grows)}")
    N = 20011
    for F in (2, 15, 24, 32):
        for D in (3, 8, 11):
            g = torch.Generator().manual_seed(F * 1000 + D + 7)
            rs = (F * D + 1 + 3) // 4 * 4
            tab = torch.zeros(N, rs)
            tab[:, :F * D + 1] = torch.randn(N, F * D + 1, generator=g) * 0.2
            x = torch.randint(0, N, (B, F), generator=g)
            x[0, 0] = N + 5
            tab, x = tab.to(dev), x.to(dev)
            t = _lib.Table(tab.data_ptr(), N, rs, F * D, 0, F * D, 0)
            bias = torch.tensor([0.125], device=dev)
            logit = torch.zeros(B, device=dev)
            pctr = torch.zeros(B, device=dev)
            part = torch.zeros(B * F, rs, device=dev)
            _lib.check(lib.rlctr_ffm_fwd(x.data_ptr(), C.byref(t), bias.data_ptr(), logit.data_ptr(), pctr.data_ptr(), 1, part.data_ptr(),
                                         B, F, D, st), "rlctr_ffm_fwd")
            lines.append(f"ffm_fwd F={F} D={D} logit {digest(logit)}")
            lines.append(f"ffm_fwd F={F} D={D} pctr {digest(pctr)}")
            lines.append(f"ffm_fwd F={F} D={D} partners {digest(part)}")
    torch.cuda.synchronize()
    with open(out, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    print(len(lines), "digests ->", out)


if __name__ == "__main__":
    main(sys.argv[1])
