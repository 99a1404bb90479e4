"""CPU oracle: flow fitting of the reference, restated in numpy with a hand-derived backward pass.

TEST INFRASTRUCTURE ONLY.  Only tests/ may import this module; the product package (nnest_b200) never does.

Restates (no code shared with) the reference:
  * nnest/trainer.py:384-403  Trainer._train: per mini-batch  data = x + jitter * randn;  loss = -mean(log_probs);
                              backward; optimizer.step(); returns sum(batch losses) / len(dataset)
  * nnest/trainer.py:405-418  Trainer._validate: -mean(log_probs(x_valid)) / len(x_valid)
  * nnest/networks.py:71-76   log_probs = N(0, I).log_prob(forward(x)) + log_det
  * nnest/networks.py:289-298 CouplingLayer.forward: z = x * exp(log_s) + t on the un-masked half
  * torch.optim.Adam (trainer.py:119-120: lr, weight_decay = 1e-6, default betas / eps), single-tensor update rule
The reference differentiates with autograd; this file writes the same derivatives out so that a CUDA kernel can be
checked layer by layer.  Arithmetic is float64 (the goldens recorded from the reference in float32 agree to ~1e-6).
Parity is pinned against the real reference: tests/golden/make_golden_train.py, tests/test_oracle_train.py.

Parameters are handled as one flat vector in netG.state_dict() order (block 0 scale net: W1 (H,d), b1, [W2 (H,H), b2]
x L, W3 (d,H), b3; block 0 translate net; block 1 ...), the layout nnb_set_flow / nnb_train_epoch use.
"""
import numpy as np


def net_floats(d, H, L):
    return H * d + H + L * (H * H + H) + d * H + d


def flatten_state_dict(sd, blocks):
    parts = []
    for k in range(blocks):
        for net in ('scale_net', 'translate_net'):
            j = 0
            while 'flow.flows.%d.%s.%d.weight' % (k, net, 2 * j) in sd:
                parts.append(np.asarray(sd['flow.flows.%d.%s.%d.weight' % (k, net, 2 * j)]).ravel())
                parts.append(np.asarray(sd['flow.flows.%d.%s.%d.bias' % (k, net, 2 * j)]).ravel())
                j += 1
    return np.concatenate(parts)


def _split_net(v, d, H, L):
    """views of one net's flat parameters: list of (W, b)"""
    out, o = [], 0
    for (r, c) in [(H, d)] + [(H, H)] * L + [(d, H)]:
        W = v[o:o + r * c].reshape(r, c)
        o += r * c
        b = v[o:o + r]
        o += r
        out.append((W, b))
    return out


def _act(kind, v):
    return np.tanh(v) if kind == 0 else np.maximum(v, 0.0)


def _dact(kind, h):
    return 1.0 - h * h if kind == 0 else (h > 0).astype(h.dtype)


def _mlp_forward(layers, kind, xin):
    acts = [xin]
    h = xin
    for (W, b) in layers[:-1]:
        h = _act(kind, h @ W.T + b)
        acts.append(h)
    W, b = layers[-1]
    return h @ W.T + b, acts


def _mlp_backward(layers, glayers, kind, acts, dout):
    """accumulates parameter gradients into glayers, returns d loss / d input"""
    W, b = layers[-1]
    gW, gb = glayers[-1]
    gW += dout.T @ acts[-1]
    gb += dout.sum(0)
    dh = dout @ W
    for li in range(len(layers) - 2, -1, -1):
        dpre = dh * _dact(kind, acts[li + 1])
        W, b = layers[li]
        gW, gb = glayers[li]
        gW += dpre.T @ acts[li]
        gb += dpre.sum(0)
        dh = dpre @ W
    return dh


def nll_and_grad(flat, x, d, H, L, B, want_grad=True, dtype=np.float64):
    """-log p(x) per sample (n,), and the gradient of mean(-log p) with respect to the flat parameters.
    dtype=np.float32 runs the same arithmetic in float32: its distance from the float64 result measures how well a float32
    implementation can do on the given inputs."""
    flat = np.asarray(flat, dtype=dtype)
    x = np.asarray(x, dtype=dtype)
    n = x.shape[0]
    nP = net_floats(d, H, L)
    nets = [(_split_net(flat[(2 * k) * nP:(2 * k + 1) * nP], d, H, L),
             _split_net(flat[(2 * k + 1) * nP:(2 * k + 2) * nP], d, H, L)) for k in range(B)]
    saved = []
    y = x
    ld = np.zeros(n, dtype=dtype)
    for k in range(B):
        mask = ((np.arange(d) + k) % 2).astype(dtype)
        xm = y * mask
        s, acts_s = _mlp_forward(nets[k][0], 0, xm)
        t, acts_t = _mlp_forward(nets[k][1], 1, xm)
        s = s * (1 - mask)
        t = t * (1 - mask)
        z = y * np.exp(s) + t
        saved.append((y, mask, s, acts_s, acts_t))
        ld += s.sum(1)
        y = z
    nll = 0.5 * (y * y).sum(1) + dtype(0.5 * d * np.log(2 * np.pi)) - ld
    if not want_grad:
        return nll, None
    grad = np.zeros_like(flat)
    gnets = [(_split_net(grad[(2 * k) * nP:(2 * k + 1) * nP], d, H, L),
              _split_net(grad[(2 * k + 1) * nP:(2 * k + 2) * nP], d, H, L)) for k in range(B)]
    gy = y / n
    for k in range(B - 1, -1, -1):
        xin, mask, s, acts_s, acts_t = saved[k]
        ds = (gy * xin * np.exp(s) - 1.0 / n) * (1 - mask)
        dt = gy * (1 - mask)
        dxm = _mlp_backward(nets[k][0], gnets[k][0], 0, acts_s, ds) + \
            _mlp_backward(nets[k][1], gnets[k][1], 1, acts_t, dt)
        gy = gy * np.exp(s) + dxm * mask
    return nll, grad


def relu_margin(flat, x, d, H, L, B):
    """Per sample (n,), the smallest |pre-activation| of any ReLU unit of the translate nets.  The gradient jumps where
    one crosses 0, so where the margin is within rounding error a float32 implementation and this oracle may differ by
    the size of the jump."""
    flat = np.asarray(flat, dtype=np.float64)
    y = np.asarray(x, dtype=np.float64)
    nP = net_floats(d, H, L)
    margin = np.full(y.shape[0], np.inf)
    for k in range(B):
        mask = ((np.arange(d) + k) % 2).astype(np.float64)
        s, _ = _mlp_forward(_split_net(flat[(2 * k) * nP:(2 * k + 1) * nP], d, H, L), 0, y * mask)
        layers = _split_net(flat[(2 * k + 1) * nP:(2 * k + 2) * nP], d, H, L)
        h = y * mask
        for (W, b) in layers[:-1]:
            pre = h @ W.T + b
            margin = np.minimum(margin, np.abs(pre).min(1))
            h = np.maximum(pre, 0.0)
        W, b = layers[-1]
        y = y * np.exp(s * (1 - mask)) + (h @ W.T + b) * (1 - mask)
    return margin


class Adam(object):
    """torch.optim.Adam, single-tensor rule, L2 weight decay added to the gradient."""

    def __init__(self, n, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.m, self.v, self.step = np.zeros(n), np.zeros(n), 0
        self.lr, self.betas, self.eps, self.wd = lr, betas, eps, weight_decay

    def update(self, w, g):
        b1, b2 = self.betas
        self.step += 1
        g = g + self.wd * w
        self.m += (g - self.m) * (1 - b1)
        self.v = self.v * b2 + (1 - b2) * g * g
        bc1, bc2 = 1 - b1 ** self.step, 1 - b2 ** self.step
        return w - (self.lr / bc1) * self.m / (np.sqrt(self.v) / np.sqrt(bc2) + self.eps)


def train_epoch(flat, opt, x_train, batch, d, H, L, B, jitter=0.0, noise=None):
    """Trainer._train over x_train in the given order.  Returns (new flat parameters, train loss)."""
    n = x_train.shape[0]
    total = 0.0
    for s in range(0, n, batch):
        xb = np.asarray(x_train[s:s + batch], dtype=np.float64)
        if jitter:
            xb = xb + jitter * np.asarray(noise[s:s + batch], dtype=np.float64)
        nll, g = nll_and_grad(flat, xb, d, H, L, B)
        total += nll.mean()
        flat = opt.update(flat, g)
    return flat, total / n


def validate(flat, x_valid, d, H, L, B):
    nll, _ = nll_and_grad(flat, x_valid, d, H, L, B, want_grad=False)
    return nll.mean() / x_valid.shape[0]
