"""CPU oracle for the decoder-query + PDE-residual hot path of flyakon/DeepPhysiNet.

TEST INFRASTRUCTURE ONLY.  This module is a plain-PyTorch (CPU, fp32 or fp64) restatement of
the reference's algorithm for the path named in BASELINE.json:north_star.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import it; the
product (deepphysinet_b200/) never does and has no CPU fallback.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md section 4), so this
oracle is pinned by running the UNMODIFIED reference in the build container
(oracle/ref_harness.py + oracle/make_golden.py) and committing the resulting vectors under
tests/golden/; tests/test_oracle_golden.py checks this file against them on every run, and
oracle/make_golden.py re-generates the vectors (and with them the live comparison) when /root/reference is mounted.

Every function cites the reference lines it follows (paths relative to /root/reference).
It keeps the reference's structure on purpose - six separate coordinate nets, one
autograd.grad(create_graph=True) call per derivative the reference takes (28 per call), MSE
per residual - so that timing it on the host cores is a fair "port" of the reference's CPU path.
"""
from __future__ import annotations

import math
from typing import Dict, Sequence

import torch

# Output order of PhysicsNet.forward (DeepPhysiNet/model/physics_net.py:49-55): net i reads
# coord_data[:, i] as its residual skip.  Module attribute names per physics_net.py:25-30.
NET_NAMES = ("U_net", "V_net", "P_net", "T_net", "q_net", "rio_net")
OBS_KEYS = ("u10", "v10", "pres", "t2", "q2", "rio")  # interface_physics.py:256-261

# configs/DeepPhysiNet_NCEP_cfg.py:64-83 (obs_norm_cfg): (mean, std, lo, hi)
OBS_NORM = {
    "u10": (0.14507186950562942, 3.0050219075895894, -500.0, 500.0),
    "v10": (-0.17325370241478535, 3.006602165591562, -500.0, 500.0),
    "pres": (89741.36105771353, 13296.749084125422, 10000.0, 500000.0),
    "t2": (283.58054561520305, 15.583177935722373, 50.0, 500.0),
    "q2": (0.007909478276582905, 0.006304067969976075, 1e-6, 10.0),
    "rio": (1.0966503643401704, 0.15166081218127583, 1e-6, 10.0),
}
# configs/DeepPhysiNet_NCEP_cfg.py:139-148
LOSS_FACTOR = dict(motion_u_factor=1.0e3, motion_v_factor=1.0e3, continuous_factor=1.0e10,
                   energy_factor=1e1, vapor_factor=1.0e14, gas_factor=1.0e-7)
TERM_NAMES = ("motion_u", "motion_v", "continuous", "energy", "vapor", "gas")


def freq_bands(n_freqs: int, max_freq: float = 4.0) -> torch.Tensor:
    """utils/position_encoding.py:26-27 - the buffer is built in fp32 and stays fp32-valued."""
    return 2.0 ** torch.linspace(0.0, max_freq, steps=n_freqs, dtype=torch.float32)


def sine_cos_pe(v: torch.Tensor, n_freqs: int) -> torch.Tensor:
    """utils/position_encoding.py:35-50 with include_input=False.
    out[..., f*2C + k*C + c] = fn_k(v[..., c] * band_f), fn_0 = sin, fn_1 = cos."""
    bands = freq_bands(n_freqs).to(device=v.device, dtype=v.dtype)
    arg = v[..., None, :] * bands[:, None]                 # [..., F, C]
    emb = torch.stack((torch.sin(arg), torch.cos(arg)), dim=-2)  # [..., F, 2, C]
    return emb.reshape(v.shape[:-1] + (-1,))


def encoding_coord(x, y, t, dx, dy, lat_size, lon_size, pred_t_span):
    """interface/interface_physics.py:322-332."""
    xn = x / dx / (lon_size - 1)
    yn = y / dy / (lat_size - 1)
    tn = t / pred_t_span
    return sine_cos_pe(torch.cat((xn, yn, tn), dim=1), 32)


def hyper_weights(meta_out: torch.Tensor, P: Dict[str, torch.Tensor], token_num=256, in_ch=192, hid=256):
    """model/variable_net.py:57-65: the first two decoder layers are generated from encoder tokens."""
    m = meta_out.reshape(-1, meta_out.shape[-1])[:token_num]                    # [tok, d]
    g1 = torch.nn.functional.linear(m.T, P["coord_input_fc.weight"], P["coord_input_fc.bias"])    # [d, 193]
    g2 = torch.nn.functional.linear(m.T, P["coord_hidden_fc.weight"], P["coord_hidden_fc.bias"])  # [d, 257]
    return g1[:, :in_ch], g1[:, in_ch], g2[:, :hid], g2[:, hid]


def lead_embedding(fore_h: torch.Tensor, P: Dict[str, torch.Tensor], in_ch=192):
    """model/variable_net.py:75-78: fore_h [1,1,1] -> squeeze(-1) -> PE(1, 96 freqs) -> fore_h_fc."""
    fh = fore_h.reshape(1, 1)
    return torch.nn.functional.linear(sine_cos_pe(fh, in_ch // 2), P["fore_h_fc.weight"], P["fore_h_fc.bias"])


def decoder_net(coord_pe, coord_data, ref, w1, b1, w2, b2, e, P):
    """model/variable_net.py:67-87 for one net, given generated weights and lead embedding e."""
    h = torch.relu(coord_pe @ w1.T + b1)
    h = h @ w2.T + b2
    d = torch.nn.functional.linear(sine_cos_pe(coord_data, 16), P["data_input_fc.weight"], P["data_input_fc.bias"])
    c = h + d + e
    r = torch.nn.functional.linear(torch.relu(torch.nn.functional.linear(c, P["cat_fc1.fc.0.weight"], P["cat_fc1.fc.0.bias"])),
                                   P["cat_fc1.fc.2.weight"], P["cat_fc1.fc.2.bias"])
    s = (r + c) + c                                       # ResMLP skip (:23-24) plus the extra skip (:85)
    return torch.nn.functional.linear(s, P["out_fc.weight"], P["out_fc.bias"]) + ref


def split_params(state: Dict[str, torch.Tensor]) -> Dict[str, Dict[str, torch.Tensor]]:
    """physics_net state_dict -> {net_name: {local_key: tensor}} for the six decoder nets."""
    out = {n: {} for n in NET_NAMES}
    for k, v in state.items():
        head, _, tail = k.partition(".")
        if head in out:
            out[head][tail] = v
    return out


def stack_generated(meta_out, fore_h, params):
    """Everything the fused operator takes as (differentiable) tensor input, stacked over the six
    nets in NET_NAMES order: generated W1,b1,W2,b2 (variable_net.py:57-65), lead embedding e
    (:75-78) and the static decoder parameters (views of `params`, so autograd reaches them)."""
    gen = [hyper_weights(meta_out, params[n]) for n in NET_NAMES]
    W = dict(W1=torch.stack([g[0] for g in gen]), b1=torch.stack([g[1] for g in gen]),
             W2=torch.stack([g[2] for g in gen]), b2=torch.stack([g[3] for g in gen]),
             e=torch.stack([lead_embedding(fore_h, params[n]).reshape(-1) for n in NET_NAMES]))
    for key, name in (("Wd", "data_input_fc.weight"), ("bd", "data_input_fc.bias"),
                      ("Wa", "cat_fc1.fc.0.weight"), ("ba", "cat_fc1.fc.0.bias"),
                      ("Wb", "cat_fc1.fc.2.weight"), ("bb", "cat_fc1.fc.2.bias"),
                      ("wo", "out_fc.weight"), ("bo", "out_fc.bias")):
        W[key] = torch.stack([params[n][name].reshape(-1) if key in ("wo", "bo") else params[n][name]
                              for n in NET_NAMES])
    W["bo"] = W["bo"].reshape(6)
    return W


def _net_params(W, k):
    return {"data_input_fc.weight": W["Wd"][k], "data_input_fc.bias": W["bd"][k],
            "cat_fc1.fc.0.weight": W["Wa"][k], "cat_fc1.fc.0.bias": W["ba"][k],
            "cat_fc1.fc.2.weight": W["Wb"][k], "cat_fc1.fc.2.bias": W["bb"][k],
            "out_fc.weight": W["wo"][k].reshape(1, -1), "out_fc.bias": W["bo"][k].reshape(1)}


def decode_generated(coord_pe, coord_data, W):
    """model/physics_net.py:49-55 on stacked tensors: net k takes coord_data[:, k] as residual skip."""
    return [decoder_net(coord_pe, coord_data, coord_data[:, k:k + 1], W["W1"][k], W["b1"][k], W["W2"][k],
                        W["b2"][k], W["e"][k], _net_params(W, k)) for k in range(6)]


def physics_net_decode(meta_out, coord_pe, coord_data, fore_h, params):
    """model/physics_net.py:41-55 minus the encoder call (meta_out is given)."""
    return decode_generated(coord_pe, coord_data, stack_generated(meta_out, fore_h, params))


def norm_of(consts) -> Dict[str, tuple]:
    """OBS_NORM-shaped {key: (mean, std, lo, hi)} of a deepphysinet_b200.config.PhysicsConsts."""
    return {k: (consts.mean[i], consts.std[i], consts.lo[i], consts.hi[i]) for i, k in enumerate(OBS_KEYS)}


def inverse_norm(outs: Sequence[torch.Tensor], with_clip: bool, norm: Dict[str, tuple] = OBS_NORM):
    """interface/interface_physics.py:232-262: mean_norm de-normalisation; clip on P,T,q,rio only.
    norm: {key: (mean, std, lo, hi)} of the config's obs_norm_cfg (default: the reference config)."""
    res = []
    for i, key in enumerate(OBS_KEYS):
        mu, sd, lo, hi = norm[key]
        v = outs[i] * sd + mu
        if with_clip and i >= 2:
            v = torch.clip(v, lo, hi)
        res.append(v)
    return res


def _grad(yv, xv):
    """interface/interface_physics.py:90-95."""
    return torch.autograd.grad(yv, xv, grad_outputs=torch.ones_like(yv), create_graph=True,
                               only_inputs=True, allow_unused=False)[0]


def _mse(a, b):
    return torch.mean((a - b) ** 2)                        # nn.MSELoss() via losses/builder.py:10


def saturation_q(p, T):
    """interface/interface_physics.py:181-185."""
    tc = T - 273.15
    e_s = 6.112 * torch.exp(17.67 * tc / (tc + 243.5)) * 100
    return 0.622 * e_s / (p - 0.378 * e_s)


def residual_losses(x, y, t, f, u, v, p, T, q, rio, factors=LOSS_FACTOR, c_p=1005, L=2.5e6, R_v=461.5, R_d=287):
    """The six loss terms of interface/interface_physics.py:97-179, in the order of TERM_NAMES,
    taking every derivative the reference takes (duplicates included)."""
    # :97-104
    u_t, u_x, u_y, p_x = _grad(u, t), _grad(u, x), _grad(u, y), _grad(p, x)
    l_u = _mse(u_t + u * u_x + v * u_y + p_x / rio, f * v) * factors["motion_u_factor"]
    # :106-114
    v_t, v_x, v_y, p_y = _grad(v, t), _grad(v, x), _grad(v, y), _grad(p, y)
    l_v = _mse(v_t + u * v_x + v * v_y + p_y / rio, -f * u) * factors["motion_v_factor"]
    # :116-124
    u_x, v_y = _grad(u, x), _grad(v, y)
    r_t, r_x, r_y = _grad(rio, t), _grad(rio, x), _grad(rio, y)
    cont = r_t + u * r_x + v * r_y + rio * u_x + rio * v_y
    l_c = _mse(cont, torch.zeros_like(cont)) * factors["continuous_factor"]
    # :126-144
    T_t, T_x, T_y = _grad(T, t), _grad(T, x), _grad(T, y)
    p_t, p_x, p_y = _grad(p, t), _grad(p, x), _grad(p, y)
    q_t, q_x, q_y = _grad(q, t), _grad(q, x), _grad(q, y)
    en = c_p * (T_t + u * T_x + v * T_y) - (p_t + u * p_x + v * p_y) / (rio + 1e-6) + L * (q_t + u * q_x + v * q_y)
    l_e = _mse(en, torch.zeros_like(en)) * factors["energy_factor"]
    # :146-175
    p_t, p_x, p_y = _grad(p, t), _grad(p, x), _grad(p, y)
    q_t, q_x, q_y = _grad(q, t), _grad(q, x), _grad(q, y)
    q_s = saturation_q(p, T).detach()
    q_s = torch.maximum(q_s, torch.ones_like(q_s) * 1e-6)
    dp = p_t + u * p_x + v * p_y
    delta = torch.where(torch.logical_and(dp < 0, torch.ge(q, q_s)), torch.ones_like(dp), torch.zeros_like(dp)).detach()
    R = (1 + 0.608 * q) * R_d
    F = ((L * R - c_p * R_v * T) / (c_p * R_v + T * T + L * L * q_s) * q_s * T).detach()
    vap = -dp * delta * F / (p + 1e-6) + (q_t + u * q_x + v * q_y)
    l_q = _mse(vap, torch.zeros_like(vap)) * factors["vapor_factor"]
    # :177-179
    l_g = _mse(p, rio * (1 + 0.608 * q) * R_d * T) * factors["gas_factor"]
    return [l_u, l_v, l_c, l_e, l_q, l_g]


def place_generated(x, y, t, f, coord_data, W, *, dx=27000.0, dy=27000.0, lat_size=145, lon_size=257,
                    pred_t_span=86400.0, with_clip=True, factors=LOSS_FACTOR, norm=OBS_NORM, c_p=1005, L=2.5e6, R_v=461.5, R_d=287,
                    return_fields=False):
    """interface/interface_physics.py:271-320 for ONE sample, from the fused operator's own inputs.

    x, y, t, f: [N,1]; coord_data [N,6]; W = stack_generated(...) (tensors may require grad).
    norm, factors, c_p, L, R_v, R_d: the constants of inverse_norm and residual_losses (defaults: the reference's).
    Returns (total, [6 terms]) and, with return_fields, also (vals [N,6] physical, jac [N,6,3] d/dx,dy,dt).
    """
    x = x.detach().clone().requires_grad_(True)
    y = y.detach().clone().requires_grad_(True)
    t = t.detach().clone().requires_grad_(True)
    pe = encoding_coord(x, y, t, dx, dy, lat_size, lon_size, pred_t_span)
    outs = decode_generated(pe, coord_data, W)
    u, v, p, T, q, rio = inverse_norm(outs, with_clip, norm)
    terms = residual_losses(x, y, t, f, u, v, p, T, q, rio, factors, c_p, L, R_v, R_d)
    total = terms[0] + terms[1] + terms[3] + terms[2] + terms[4] + terms[5]   # summation order of :301
    if not return_fields:
        return total, terms
    phys = (u, v, p, T, q, rio)
    vals = torch.cat([a.detach() for a in phys], dim=1)
    jac = torch.stack([torch.cat([torch.autograd.grad(a.sum(), c, retain_graph=True)[0] for c in (x, y, t)], dim=1)
                       for a in phys], dim=1)
    return total, terms, vals, jac.detach()


def place_one_batch(x, y, t, f, coord_data, fore_h, meta_out, params, **kw):
    """Same, from the encoder output and the physics_net parameters (split_params(state_dict))."""
    return place_generated(x, y, t, f, coord_data, stack_generated(meta_out, fore_h, params), **kw)


def place_batch(samples, params_of, **kw):
    """SURVEY D4: the reference is structurally batch-1; batch B = B independent samples, loss = mean
    over samples (the DDP semantics of interface_physics.py:899-907,1056)."""
    totals = [place_one_batch(*s, params_of, **kw)[0] for s in samples]
    return sum(totals) / len(totals)


# ---------------------------------------------------------------------------------------------
# Synthetic inputs (SURVEY.md 8(d)); mirrors dataset/physics_dataset.py:442-446,492-496,521-526.
# Deterministic given the generator; used identically by tests and bench so CPU and GPU arms see
# the same numbers.
# ---------------------------------------------------------------------------------------------
def synthetic_points(n, gen: torch.Generator, *, dx=27000.0, dy=27000.0, lat_size=145, lon_size=257,
                     begin_lat=18.0, deg_per_cell=0.25, dtype=torch.float32):
    xg = torch.rand(n, 1, generator=gen, dtype=torch.float64) * (lon_size - 1)
    yg = torch.rand(n, 1, generator=gen, dtype=torch.float64) * (lat_size - 1)
    th = torch.randint(0, 25, (n, 1), generator=gen).to(torch.float64)
    lat = begin_lat + yg * deg_per_cell
    f = 2 * 7.29e-5 * torch.sin(lat / 180 * math.pi)
    coord_data = 0.5 * torch.randn(n, 6, generator=gen, dtype=torch.float64)
    return ((xg * dx).to(dtype), (yg * dy).to(dtype), (th * 3600).to(dtype), f.to(dtype), coord_data.to(dtype))
