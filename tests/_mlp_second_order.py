"""TEST INFRASTRUCTURE ONLY: the float64 reference of the SDF network's second derivative (the eikonal term of
hmsdf.py:856-880: autograd.grad(sdf, x, create_graph=True), then a loss on that gradient), built on the first-order oracle
oracle/mlp_oracle.py (its `forward` cache).  Pinned against torch float64 double backward and the live reference module in
tests/test_mlp_oracle_second_order.py; the GPU tests of tests/test_zzzzzzzz_mlp_second_order.py compare against it."""
from __future__ import annotations

import numpy as np

from oracle.mlp_oracle import BETA, THRESHOLD, embed_backward, softplus_grad


def softplus_grad2(z):
    """d^2 softplus / dz^2, zero past the threshold (torch's softplus_double_backward)."""
    t = BETA * z
    s = 1.0 / (1.0 + np.exp(-np.minimum(t, THRESHOLD)))
    return np.where(t > THRESHOLD, 0.0, BETA * s * (1.0 - s))


def embed_tangent(x, n_freq, v):
    """E'(x) v: the directional derivative of the encoding along v (M,3)."""
    x, v = np.asarray(x, dtype=np.float64), np.asarray(v, dtype=np.float64)
    out = [v]
    for k in range(n_freq):
        f = 2.0 ** k
        out += [f * np.cos(f * x) * v, -f * np.sin(f * x) * v]
    return np.concatenate(out, -1)


def embed_second_backward(x, n_freq, v, g_emb):
    """E''(x)[v]^T g_emb: the derivative of embed_backward(x, n_freq, g_emb) with respect to x along v (diagonal per
    coordinate)."""
    x, v = np.asarray(x, dtype=np.float64), np.asarray(v, dtype=np.float64)
    g = np.zeros_like(x)
    for k in range(n_freq):
        f = 2.0 ** k
        g -= f * f * v * (np.sin(f * x) * g_emb[:, 3 + 6 * k:6 + 6 * k] + np.cos(f * x) * g_emb[:, 6 + 6 * k:9 + 6 * k])
    return g


def second_order(cache, g_out, v):
    """Second derivative of the network: with g_x = backward(cache, g_out)[0] and s = sum(v * g_x) for an upstream v (M,3),
    -> (ds/dx (M,3), [ds/dweight...], [ds/dbias...], y_dot) where y_dot = J(x) v (M, d_out) is ds/dg_out.  The output
    layer's bias does not enter g_x: its entry is zeros (torch reports None).  Tangent pass along x' = v, then the adjoint
    of the first backward pass, with softplus' and softplus'' of the float64 pre-activations."""
    w, inputs, pre = cache["w"], cache["inputs"], cache["pre"]
    x, n_freq, skip_in = cache["x"], cache["n_freq"], cache["skip_in"]
    n_layers = len(w)
    n_hidden = n_layers - 2
    e = cache["emb"].shape[1]
    gy = np.asarray(g_out, dtype=np.float64)
    v = np.asarray(v, dtype=np.float64)
    wide = [1 <= li <= n_hidden and (li - 1) in skip_in for li in range(n_layers)]
    # first backward: lam[li] = gradient at the output a_li of hidden layer li, delta[li] at its pre-activation
    lam, delta = [None] * (n_hidden + 1), [None] * (n_hidden + 1)
    g_emb = np.zeros_like(cache["emb"])
    lam[n_hidden] = gy @ w[-1]
    for li in range(n_hidden, -1, -1):
        delta[li] = lam[li] * softplus_grad(pre[li])
        g_in = delta[li] @ w[li]
        if wide[li]:
            g_emb += g_in[:, -e:]
            g_in = g_in[:, :-e]
        if li == 0:
            g_emb += g_in
        else:
            lam[li - 1] = g_in
    # tangent pass
    e_dot = embed_tangent(x, n_freq, v)
    h_dot, z_dot = [], []
    h = e_dot
    for li in range(n_hidden + 1):
        if wide[li]:
            h = np.concatenate([h, e_dot], -1)
        h_dot.append(h)
        z_dot.append(h @ w[li].T)
        h = z_dot[li] * softplus_grad(pre[li])
    y_dot = h @ w[-1].T
    gw, gb = [None] * n_layers, [None] * n_layers
    gw[-1], gb[-1] = gy.T @ h, np.zeros(w[-1].shape[0])
    # adjoint of the first backward pass; mu = gradient at the pre-activation of hidden layer li
    g_bar = np.zeros_like(cache["emb"])
    mu = lam[n_hidden] * softplus_grad2(pre[n_hidden]) * z_dot[n_hidden]
    for li in range(n_hidden, -1, -1):
        gw[li] = mu.T @ inputs[li] + delta[li].T @ h_dot[li]
        gb[li] = mu.sum(0)
        p = mu @ w[li]
        if wide[li]:
            g_bar += p[:, -e:]
            p = p[:, :-e]
        if li == 0:
            g_bar += p
        else:
            mu = p * softplus_grad(pre[li - 1]) + lam[li - 1] * softplus_grad2(pre[li - 1]) * z_dot[li - 1]
    g_x = embed_backward(x, n_freq, g_bar) + embed_second_backward(x, n_freq, v, g_emb)
    return g_x, gw, gb, y_dot
