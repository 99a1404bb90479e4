"""CPU oracle: RealNVP / affine-coupling flow of the reference, restated in numpy float32 (and, with dtype=np.float64,
in float64 on the same float32 weights: a reference whose own rounding is negligible next to a float32 kernel's).

TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference leg may import this module; the product package (nnest_b200) never does.

Restates (no code shared with) the reference:
  * nnest/networks.py:24-42   NormalizingFlow.forward / inverse  (layer loop, log_det accumulation)
  * nnest/networks.py:248-309 CouplingLayer (s-net tanh, t-net relu, no activation on the last Linear)
  * nnest/networks.py:312-325 ScaleLayer (scale='constant')
  * nnest/networks.py:328-347 SingleSpeedNVP (block k uses mask (arange(d)+k) % 2)
Parity is pinned against the real reference run in the build container: see
tests/golden/make_golden.py and tests/test_oracle_golden.py.
"""
import numpy as np

F32 = np.float32


class NVPWeights(object):
    """Weights of a SingleSpeedNVP, in the reference's own (out, in) nn.Linear layout.

    blocks[k] = {'scale': [(W, b), ...] or None, 'translate': [(W, b), ...], 'const_scale': float or None}
    """

    def __init__(self, d, hidden, num_layers, num_blocks, blocks, translate_only=False):
        self.d = int(d)
        self.hidden = int(hidden)
        self.num_layers = int(num_layers)
        self.num_blocks = int(num_blocks)
        self.blocks = blocks
        self.translate_only = bool(translate_only)

    def mask(self, k):
        # networks.py:333-346 : mask starts as arange(d) % 2 and is flipped after every block
        return ((np.arange(self.d) + k) % 2).astype(F32)

    @classmethod
    def from_state_dict(cls, sd, d, scale=''):
        """sd: mapping name -> array-like, names as produced by netG.state_dict()
        ('flow.flows.<i>.scale_net.<2j>.weight', ...).  scale: the reference's `scale` kwarg."""
        sd = {k: np.asarray(v.detach().cpu().numpy() if hasattr(v, 'detach') else v, dtype=F32)
              for k, v in sd.items()}
        translate_only = scale in ('translate', 'constant')
        stride = 2 if scale == 'constant' else 1
        idx = sorted({int(k.split('.')[2]) for k in sd if k.startswith('flow.flows.')})
        num_blocks = (max(idx) + 1 + stride - 1) // stride
        blocks = []
        for k in range(num_blocks):
            fi = k * stride
            blk = {'scale': None, 'translate': None, 'const_scale': None}
            for net in ('scale', 'translate'):
                if net == 'scale' and translate_only:
                    continue
                layers = []
                j = 0
                while 'flow.flows.%d.%s_net.%d.weight' % (fi, net, 2 * j) in sd:
                    layers.append((sd['flow.flows.%d.%s_net.%d.weight' % (fi, net, 2 * j)],
                                   sd['flow.flows.%d.%s_net.%d.bias' % (fi, net, 2 * j)]))
                    j += 1
                blk[net] = layers
            if scale == 'constant':
                blk['const_scale'] = float(sd['flow.flows.%d.scale' % (fi + 1)])
            blocks.append(blk)
        nl = len(blocks[0]['translate']) - 2
        hidden = blocks[0]['translate'][0][0].shape[0]
        return cls(d, hidden, nl, num_blocks, blocks, translate_only)

    @classmethod
    def random(cls, d, hidden=16, num_layers=1, num_blocks=3, seed=0, gain=1.0, scale=''):
        """nn.Linear-style default init U(-1/sqrt(fan_in), 1/sqrt(fan_in)) from a numpy generator
        (used where torch is not wanted; distribution only, not torch's stream).  scale: the reference's `scale` kwarg;
        'constant' draws each block's ScaleLayer parameter from U(-0.5, 0.5), rounded to float32."""
        assert scale in ('', 'translate', 'constant')
        translate_only = scale != ''
        rng = np.random.default_rng(seed)

        def lin(o, i):
            b = gain / np.sqrt(i)
            return (rng.uniform(-b, b, size=(o, i)).astype(F32), rng.uniform(-b, b, size=(o,)).astype(F32))

        blocks = []
        for _ in range(num_blocks):
            blk = {'scale': None, 'translate': None, 'const_scale': None}
            for net in ('scale', 'translate'):
                if net == 'scale' and translate_only:
                    continue
                layers = [lin(hidden, d)] + [lin(hidden, hidden) for _ in range(num_layers)] + [lin(d, hidden)]
                blk[net] = layers
            if scale == 'constant':
                blk['const_scale'] = float(F32(rng.uniform(-0.5, 0.5)))
            blocks.append(blk)
        return cls(d, hidden, num_layers, num_blocks, blocks, translate_only)

    def flat(self):
        """Flat float32 buffer in the C-ABI order documented in include/nnb.h: for each block,
        scale net (absent if translate_only) then translate net, each layer weight (out*in,
        row-major) followed by its bias; then one float per block of const_scale if present."""
        out = []
        for blk in self.blocks:
            for net in ('scale', 'translate'):
                if blk[net] is None:
                    continue
                for W, b in blk[net]:
                    out.append(np.ascontiguousarray(W, dtype=F32).ravel())
                    out.append(np.ascontiguousarray(b, dtype=F32).ravel())
        if self.blocks[0]['const_scale'] is not None:
            out.append(np.array([blk['const_scale'] for blk in self.blocks], dtype=F32))
        return np.concatenate(out)


def _mlp(layers, act, v, dtype=F32):
    # networks.py:273-282 : Linear, act, [Linear, act] x L, Linear  (no activation after the last)
    h = v
    n = len(layers)
    for j, (W, b) in enumerate(layers):
        h = (h @ np.asarray(W, dtype=dtype).T + np.asarray(b, dtype=dtype)).astype(dtype)
        if j < n - 1:
            h = np.tanh(h) if act == 'tanh' else np.maximum(h, dtype(0))
    return h.astype(dtype)


def coupling_forward(w, k, x, dtype=F32):
    """networks.py:289-298"""
    blk = w.blocks[k]
    mask = w.mask(k).astype(dtype)
    masked = x * mask
    t = _mlp(blk['translate'], 'relu', masked, dtype) * (dtype(1) - mask)
    if blk['scale'] is None:
        return (x + t).astype(dtype), np.zeros(x.shape[0], dtype=dtype)
    log_s = _mlp(blk['scale'], 'tanh', masked, dtype) * (dtype(1) - mask)
    s = np.exp(log_s)
    return (x * s + t).astype(dtype), log_s.sum(-1, dtype=dtype)


def coupling_inverse(w, k, z, dtype=F32):
    """networks.py:300-309"""
    blk = w.blocks[k]
    mask = w.mask(k).astype(dtype)
    masked = z * mask
    t = _mlp(blk['translate'], 'relu', masked, dtype) * (dtype(1) - mask)
    if blk['scale'] is None:
        return (z - t).astype(dtype), np.zeros(z.shape[0], dtype=dtype)
    log_s = _mlp(blk['scale'], 'tanh', masked, dtype) * (dtype(1) - mask)
    s = np.exp(-log_s)
    return ((z - t) * s).astype(dtype), (-log_s).sum(-1, dtype=dtype)


def flow_forward(w, x, dtype=F32):
    """x (N,d) -> z (N,d), log_det (N,)   [networks.py:24-32, blocks in natural order]"""
    x = np.ascontiguousarray(x, dtype=dtype)
    ld = np.zeros(x.shape[0], dtype=dtype)
    for k in range(w.num_blocks):
        x, l = coupling_forward(w, k, x, dtype)
        ld = (ld + l).astype(dtype)
        cs = w.blocks[k]['const_scale']
        if cs is not None:  # ScaleLayer.forward networks.py:319-321 (log-det is the scalar itself)
            x = (x * np.exp(dtype(F32(cs)))).astype(dtype)
            ld = (ld + dtype(F32(cs))).astype(dtype)
    return x, ld


def flow_inverse(w, z, dtype=F32):
    """z (N,d) -> x (N,d), log_det (N,)   [networks.py:34-42, blocks reversed]"""
    z = np.ascontiguousarray(z, dtype=dtype)
    ld = np.zeros(z.shape[0], dtype=dtype)
    for k in range(w.num_blocks - 1, -1, -1):
        cs = w.blocks[k]['const_scale']
        if cs is not None:  # ScaleLayer.inverse networks.py:323-325 (it follows block k in the list)
            z = (z * np.exp(-dtype(F32(cs)))).astype(dtype)
            ld = (ld - dtype(F32(cs))).astype(dtype)
        z, l = coupling_inverse(w, k, z, dtype)
        ld = (ld + l).astype(dtype)
    return z, ld
