"""Float64 model of what the single-TF32 policy kernels feed the tensor core (precision 1).

kind::tf32 MMAs read 10 explicit mantissa bits of each operand and accumulate in float32.  The kernels
build their operands as follows:
  * packed weights and layer-1 / layer-2 biases: rounded to nearest, ties away (`tf32_rna`, k_pack_tc);
  * k_policy_tc: the standardised observation X and the hidden activations are rounded the same way before
    they are stored as operands (pdx_policy_tc.cu, build_x and hidden_epilogue);
  * k_collect: X and the layer-1 activations are passed as raw float32 words; the tensor core converts them
    itself (`convert`: 'trunc' drops the low 13 bits, 'rna' rounds);
  * layer 3 (64 x 4 actor and 64 x 1 critic weights) runs in float32 on the CUDA cores, unrounded;
  * the critic's tanh is `tanh.approx.f32` (relative error below 2^-10.987, PTX ISA): the model evaluates
    the exact tanh and `tanh_bound` bounds what the approximation can add.
"""
import numpy as np

TANH_APPROX_REL = 2.0 ** -10.987


def tf32(x, mode='rna'):
    """float32 -> float32 on the tf32 grid: 'rna' = (bits + 0x1000) & ~0x1fff as tf32_rna, 'trunc' = bits & ~0x1fff."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    if mode == 'rna':
        u = u + np.uint32(0x1000)
    elif mode != 'trunc':
        raise ValueError(mode)
    return (u & np.uint32(0xFFFFE000)).view(np.float32)


def standardise32(obs, mean, std, eps):
    """The kernels' float32 standardisation (o - mean) * (1 / (std + eps)); no normaliser: o itself."""
    obs = np.asarray(obs, dtype=np.float32)
    if mean is None:
        return obs
    inv = np.float32(1.0) / (np.asarray(std, np.float32) + np.float32(eps))
    return (obs - np.asarray(mean, np.float32)) * inv


def forward(obs, mean, std, eps, pi_layers, v_layers, convert='rna'):
    """(mu [N, n_out], v [N], bound-terms) of the single-TF32 kernels in float64.  Layers: [(W [out][in], b)],
    float32 values.  The third element holds what `tanh_bound` needs."""
    x = tf32(standardise32(obs, mean, std, eps), convert).astype(np.float64)
    r = lambda a: tf32(a).astype(np.float64)
    (w1, b1), (w2, b2), (w3, b3) = pi_layers
    h = np.maximum(x @ r(w1).T + r(b1), 0.0)
    h = tf32(h.astype(np.float32), convert).astype(np.float64)
    h = np.maximum(h @ r(w2).T + r(b2), 0.0)
    mu = h @ np.asarray(w3, np.float64).T + np.asarray(b3, np.float64)
    (c1, d1), (c2, d2), (c3, d3) = v_layers
    y1 = np.tanh(x @ r(c1).T + r(d1))
    y1 = tf32(y1.astype(np.float32), convert).astype(np.float64)
    y2 = np.tanh(y1 @ r(c2).T + r(d2))
    w3c = np.asarray(c3, np.float64)[0]
    v = y2 @ w3c + float(d3[0])
    return mu, v, (y2, w3c)


def tanh_bound(terms):
    """Per row: what tanh.approx on the layer-2 activations can add to the value, its relative error times
    sum_j |y2_j| |w3c_j|.  The approximation on the layer-1 activations reaches the value through the tf32
    operands of layer 2 like any operand rounding; the tests measure that part with the TF32 term."""
    y2, w3c = terms
    return TANH_APPROX_REL * (np.abs(y2) @ np.abs(w3c))
