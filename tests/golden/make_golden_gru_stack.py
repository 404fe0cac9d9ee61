"""Golden vectors for the stacked sequence head (GruSage(gru_num_layers > 1)), produced by the reference's own layer:
`torch.nn.GRU(num_layers=L, batch_first=True)` on the CPU, called as src/models/grusage.py:160-161 does
(`gru_out, hlast = self.gru(x); x = hlast[-1]`).

    python tests/golden/make_golden_gru_stack.py      # writes tests/golden/gru_stack/*.pt

Each fixture: the constructor arguments, the state dict (every layer), x [N,T,I], an upstream gradient for the last
hidden state of the top layer, and -- in fp32 and, for adjudication, fp64 -- that hidden state and the gradients of x
and of every parameter of every layer."""
import os

import torch

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gru_stack")
# Small on purpose (every fixture well under 0.5 MB: fp32 and fp64 gradients of every layer are stored); the wider
# hidden sizes are covered by tests/test_gru_stack.py against a live CPU nn.GRU.
CASES = {"ref_hidden32_three_layers": dict(N=40, T=16, I=6, H=32, L=3),
         "ref_hidden32_wide_input": dict(N=30, T=9, I=8, H=32, L=2),
         "ref_hidden32_one_input": dict(N=25, T=5, I=1, H=32, L=2)}


def main():
    os.makedirs(OUT, exist_ok=True)
    for seed, (name, c) in enumerate(CASES.items()):
        torch.manual_seed(200 + seed)
        gru = torch.nn.GRU(input_size=c["I"], hidden_size=c["H"], num_layers=c["L"], batch_first=True)
        x = torch.randn(c["N"], c["T"], c["I"])
        up = torch.randn(c["N"], c["H"])
        fix = dict(cfg=c, state_dict={k: v.clone() for k, v in gru.state_dict().items()}, x=x, up=up)
        for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
            g = torch.nn.GRU(input_size=c["I"], hidden_size=c["H"], num_layers=c["L"], batch_first=True).to(dt)
            g.load_state_dict({k: v.to(dt) for k, v in gru.state_dict().items()})
            xi = x.detach().clone().to(dt).requires_grad_(True)
            _, hlast = g(xi)
            h = hlast[-1, :, :]
            h.backward(up.to(dt))
            fix[tag] = dict(h=h.detach().clone(), dx=xi.grad.clone(), grads={k: p.grad.clone() for k, p in g.named_parameters()})
        torch.save(fix, os.path.join(OUT, name + ".pt"))
        print(name, {k: tuple(v.shape) for k, v in fix["f32"]["grads"].items()})


if __name__ == "__main__":
    main()
