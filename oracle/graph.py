"""Generic torch-CPU executor for a layer-spec graph (oracle; test infrastructure).  Checked against oracle/model.py and
oracle/loss.py (tests/test_oracle_graph_cpu.py), which are pinned to the reference's code (tests/test_oracle_tf_shim_golden.py).

Executes the same ``Spec`` list the product's builders produce (ops INPUT / CONV / MAXPOOL / L2NORM / HEAD) with
torch.nn.functional in float32 or float64, keeping the autograd graph so that gradients of the SSD loss with respect to
every kernel / bias / gamma can be compared with the CUDA backward pass.  ``backward_teacher_forced`` differentiates the same
graph layer by layer at the activations the CUDA forward pass stored.  Conventions as in oracle/model.py.
"""
import numpy as np
import torch
import torch.nn.functional as Fn

OP_INPUT, OP_CONV, OP_MAXPOOL, OP_L2NORM, OP_HEAD = range(5)
ACT_NONE, ACT_RELU, ACT_ELU = range(3)


def make_params(specs, weights, dtype=torch.float32, requires_grad=True):
    """numpy weight dict (Keras names) -> dict of torch leaf tensors."""
    return {k: torch.tensor(np.asarray(v), dtype=dtype, requires_grad=requires_grad) for k, v in weights.items()}


def forward(specs, params, x_nhwc, n_classes_total, anchors, variances, dtype=torch.float32, bn_training=False):
    """-> y_pred (B, P, C+12) torch tensor (differentiable w.r.t. ``params``).  ``bn_training``: BatchNormalization in Keras'
    training phase (what ``fit_generator`` runs, models/keras_ssd7.py:277-309): batch mean / biased variance over (B,H,W), epsilon
    1e-3; the batch statistics are returned in ``outs['<bn>/batch_mean' | '/batch_var']`` (biased variance)."""
    outs = {}
    confs, locs = [], []
    for s in specs:
        if s.op == OP_INPUT:
            x = torch.as_tensor(np.asarray(x_nhwc), dtype=dtype)
            p = s.params
            if p.get('mean') is not None:
                x = x - torch.tensor(np.asarray(p['mean'], dtype=np.float64), dtype=dtype)
            if p.get('stddev') is not None:
                x = x / torch.tensor(np.asarray(p['stddev'], dtype=np.float64), dtype=dtype)
            if p.get('swap'):
                x = x[..., list(p['swap'])]
            outs[s.name] = x.permute(0, 3, 1, 2).contiguous()
            continue
        xin = outs[s.inp]
        if s.op == OP_CONV:
            y = _conv_pre(s, xin, params, bn_training, outs)
            if s.act == ACT_RELU:
                y = torch.relu(y)
            elif s.act == ACT_ELU:
                y = Fn.elu(y)
            outs[s.name] = y
        elif s.op == OP_MAXPOOL:
            outs[s.name] = _maxpool(s, xin)
        elif s.op == OP_L2NORM:
            outs[s.name] = _l2norm(s, xin, params)
        elif s.op == OP_HEAD:
            c, l = _head(s, xin, params, n_classes_total)
            confs.append(c)
            locs.append(l)
    conf = torch.softmax(torch.cat(confs, dim=1), dim=-1)
    loc = torch.cat(locs, dim=1)
    B, P = conf.shape[0], conf.shape[1]
    anc = torch.as_tensor(np.asarray(anchors), dtype=dtype).unsqueeze(0).expand(B, P, 4)
    var = torch.as_tensor(np.asarray(variances), dtype=dtype).view(1, 1, 4).expand(B, P, 4)
    return torch.cat([conf, loc, anc, var], dim=-1), outs


def backward_teacher_forced(specs, weights, acts, dy, n_classes_total, bn_training=False, device='cpu', fwd_err=None,
                            unrotated=None):
    """float64 gradients of ``sum(dy * y_pred)`` w.r.t. every trainable parameter, with each layer differentiated at the
    activations the CUDA forward pass stored ("teacher forcing") instead of at a float64 forward pass of its own.

    The layers are walked top-down.  Each one's local function is rebuilt in float64 from its producer's stored activation
    (a detached leaf), the gradient of its output (summed over its consumers) is applied with ``torch.autograd.grad``, and the
    gradient w.r.t. the leaf goes on to the producer.  A ReLU multiplies by ``acts[layer] > 0``, the mask the backward
    kernels read from the stored forward value, so that a pre-activation within rounding distance of 0 cannot take the other
    side of the ReLU here; max-pool routes to the first maximum of the stored input like ``pool_bwd_kernel``; L2Norm, the
    heads' softmax, ELU and BatchNormalization (batch statistics when ``bn_training``) are recomputed from the stored input.
    What is left between this and the device is the backward arithmetic itself.

    specs / weights: the model's ``Spec`` list and numpy weights (Keras names).  acts: {layer name: (B,h,w,c) activation} for
    every layer except the heads; a head's entry, if present, is its raw output (per box [C class logits | 4 offsets]) and is
    only used for the forward check.  dy: (B,P,C+12); the anchor and variance columns carry no gradient.  device: where the
    float64 arithmetic runs; each layer's temporaries are freed before the next layer.  fwd_err: optional dict, filled with
    max|local float64 forward - acts[layer]| / max|acts[layer]| per layer.  unrotated: name of a conv layer whose data
    gradient uses the kernel without the 180 degree rotation -- a deliberately wrong reference, to show that the comparison
    detects that mistake.  Returns {weight name: float64 ndarray}."""
    dev = torch.device(device)
    f64 = torch.float64
    by_name = {s.name: s for s in specs}
    dy = (dy if torch.is_tensor(dy) else torch.from_numpy(np.asarray(dy))).to(dev, f64)
    C = n_classes_total

    def load(name):
        a = acts[name]
        a = a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a))
        return a.to(dev, f64).permute(0, 3, 1, 2).contiguous()

    def record(name, got, ref):
        if fwd_err is not None:
            fwd_err[name] = float((got - ref).abs().max() / ref.abs().max().clamp(min=1e-30))

    prior_off, off = {}, 0
    for s in specs:
        if s.op == OP_HEAD:
            _, h, w, _ = np.shape(acts[s.inp])
            prior_off[s.name] = off
            off += (h + s.pad[0] + s.pad[2] - s.kh + 1) * (w + s.pad[1] + s.pad[3] - s.kw + 1) * s.n_boxes
    dout, grads = {}, {}

    def layer(s):
        g_out = None if s.op == OP_HEAD else dout.pop(s.name, None)
        if s.op != OP_HEAD and g_out is None:
            return                                          # nothing consumes this layer
        need_dx = by_name[s.inp].op != OP_INPUT
        x = load(s.inp).requires_grad_(need_dx)
        if s.op == OP_CONV:
            names = [s.name + '/kernel', s.name + '/bias']
            if getattr(s, 'bn', None):
                names += [s.bn + '/gamma', s.bn + '/beta'] if bn_training else []
        elif s.op == OP_HEAD:
            names = [s.params[k] + t for k in ('conf_name', 'loc_name') for t in ('/kernel', '/bias')]
        elif s.op == OP_L2NORM:
            names = [s.name + '/gamma']
        else:
            names = []
        p = {k: torch.tensor(np.asarray(weights[k]), dtype=f64, device=dev, requires_grad=True) for k in names}
        if getattr(s, 'bn', None) and not bn_training:
            for k in ('/gamma', '/beta', '/moving_mean', '/moving_variance'):
                p.setdefault(s.bn + k, torch.tensor(np.asarray(weights[s.bn + k]), dtype=f64, device=dev))
        z = None
        if s.op == OP_HEAD:
            c, l = _head(s, x, p, C)
            if s.name in acts:
                B, (_, h, w, _) = c.shape[0], np.shape(acts[s.name])
                fused = torch.cat([c.view(B, -1, s.n_boxes, C), l.view(B, -1, s.n_boxes, 4)], -1).reshape(B, h, w, -1)
                record(s.name, fused.detach(), torch.as_tensor(acts[s.name]).to(dev, f64))
            rows = slice(prior_off[s.name], prior_off[s.name] + c.shape[1])
            outs, g_outs = [torch.softmax(c, dim=-1), l], [dy[:, rows, :C], dy[:, rows, C:C + 4]]
        elif s.op == OP_CONV:
            z = _conv_pre(s, x, p, bn_training)
            if s.act == ACT_RELU:
                stored = load(s.name)
                record(s.name, torch.relu(z.detach()), stored)
                y = z * (stored > 0)
                del stored
            else:
                y = Fn.elu(z) if s.act == ACT_ELU else z
                record(s.name, y.detach(), load(s.name))
            outs, g_outs = [y], [g_out]
        else:
            y = _maxpool(s, x) if s.op == OP_MAXPOOL else _l2norm(s, x, p)
            record(s.name, y.detach(), load(s.name))
            outs, g_outs = [y], [g_out]
        wrt = ([x] if need_dx else []) + [p[k] for k in names] + ([z] if unrotated == s.name and need_dx else [])
        if not wrt:
            return
        res = list(torch.autograd.grad(outs, wrt, g_outs))
        del outs, g_outs, g_out
        if unrotated == s.name and need_dx:
            dz = res.pop()
            pt, pl, pb, pr = s.pad
            wf = p[s.name + '/kernel'].detach().permute(3, 2, 0, 1).flip(2, 3)
            zf = Fn.conv2d(Fn.pad(x, (pl, pr, pt, pb)), wf, stride=s.stride, dilation=s.dilation)
            res[0] = torch.autograd.grad(zf, x, dz)[0]
        if need_dx:
            dx = res.pop(0)
            dout[s.inp] = dx if s.inp not in dout else dout[s.inp] + dx
        for k, g in zip(names, res):
            grads[k] = g.cpu().numpy()

    for s in reversed(specs):
        if s.op != OP_INPUT:
            layer(s)
    return grads


def _conv_pre(s, xin, params, bn_training, outs=None):
    """A CONV layer up to its activation: convolution + bias, then BatchNormalization if the layer has one."""
    pt, pl, pb, pr = s.pad
    w = params[s.name + '/kernel'].permute(3, 2, 0, 1)
    y = Fn.conv2d(Fn.pad(xin, (pl, pr, pt, pb)), w, params[s.name + '/bias'], stride=s.stride, dilation=s.dilation)
    if getattr(s, 'bn', None) and bn_training:
        g, b = params[s.bn + '/gamma'], params[s.bn + '/beta']
        mu = y.mean(dim=(0, 2, 3)); var = y.var(dim=(0, 2, 3), unbiased=False)
        if outs is not None:
            outs[s.bn + '/batch_mean'], outs[s.bn + '/batch_var'] = mu.detach(), var.detach()
        y = (y - mu.view(1, -1, 1, 1)) / torch.sqrt(var.view(1, -1, 1, 1) + 1e-3) * g.view(1, -1, 1, 1) + b.view(1, -1, 1, 1)
    elif getattr(s, 'bn', None):        # inference-phase BatchNormalization (Keras epsilon 1e-3) between conv and activation
        g, b = params[s.bn + '/gamma'], params[s.bn + '/beta']
        mu, var = params[s.bn + '/moving_mean'], params[s.bn + '/moving_variance']
        y = (y - mu.view(1, -1, 1, 1)) / torch.sqrt(var.view(1, -1, 1, 1) + 1e-3) * g.view(1, -1, 1, 1) + b.view(1, -1, 1, 1)
    return y


def _maxpool(s, xin):
    pt, pl, pb, pr = s.pad
    return Fn.max_pool2d(Fn.pad(xin, (pl, pr, pt, pb), value=float('-inf')), (s.kh, s.kw), s.stride)


def _l2norm(s, xin, params):
    ss = torch.sum(xin * xin, dim=1, keepdim=True)
    return xin * torch.rsqrt(torch.clamp(ss, min=1e-12)) * params[s.name + '/gamma'].view(1, -1, 1, 1)


def _head(s, xin, params, n_classes_total):
    """-> (class logits (B, H*W*n_boxes, C), box offsets (B, H*W*n_boxes, 4)) in y_pred's prior order."""
    pt, pl, pb, pr = s.pad
    cn, ln = s.params['conf_name'], s.params['loc_name']
    c = Fn.conv2d(Fn.pad(xin, (pl, pr, pt, pb)), params[cn + '/kernel'].permute(3, 2, 0, 1), params[cn + '/bias'])
    l = Fn.conv2d(Fn.pad(xin, (pl, pr, pt, pb)), params[ln + '/kernel'].permute(3, 2, 0, 1), params[ln + '/bias'])
    B = c.shape[0]
    return c.permute(0, 2, 3, 1).reshape(B, -1, n_classes_total), l.permute(0, 2, 3, 1).reshape(B, -1, 4)


def ssd_loss_torch(y_true, y_pred, neg_pos_ratio=3, n_neg_min=0, alpha=1.0):
    """keras_loss_function/keras_ssd_loss.py:98-211 with torch ops -> (B,) tensor; the hard-negative mask is a constant."""
    yt = torch.as_tensor(np.asarray(y_true), dtype=y_pred.dtype)
    cls = -torch.sum(yt[:, :, :-12] * torch.log(torch.clamp(y_pred[:, :, :-12], min=1e-15)), dim=-1)
    d = yt[:, :, -12:-8] - y_pred[:, :, -12:-8]
    ad = torch.abs(d)
    loc = torch.sum(torch.where(ad < 1.0, 0.5 * d * d, ad - 0.5), dim=-1)
    neg = yt[:, :, 0]
    pos = torch.max(yt[:, :, 1:-12], dim=-1).values
    n_pos = pos.sum()
    B = yt.shape[0]
    neg_all = (cls * neg).detach()
    n_neg_losses = int(torch.count_nonzero(neg_all))
    k = min(max(int(neg_pos_ratio) * int(n_pos.item()), int(n_neg_min)), n_neg_losses)
    mask = torch.zeros_like(neg_all).reshape(-1)
    if k > 0:
        flat = neg_all.reshape(-1).double().numpy()
        order = np.lexsort((np.arange(flat.size), -flat))[:k]
        mask[torch.as_tensor(order)] = 1
    mask = mask.reshape(neg_all.shape)
    total = (torch.sum(cls * pos, -1) + torch.sum(cls * mask, -1) + alpha * torch.sum(loc * pos, -1)) / torch.clamp(n_pos, min=1.0)
    return total * B


def sgd_step(params, grads, velocity, lr, momentum, l2_reg):
    """Keras SGD (v = m*v - lr*g; w += v) with the l2 kernel regulariser's gradient 2*l2*w on kernels.  numpy dicts in/out."""
    new_p, new_v = {}, {}
    for k, w in params.items():
        g = grads[k].astype(np.float64)
        if k.endswith('/kernel'):
            g = g + 2.0 * l2_reg * w.astype(np.float64)
        v = momentum * velocity.get(k, np.zeros_like(w, dtype=np.float64)) - lr * g
        new_v[k] = v
        new_p[k] = (w.astype(np.float64) + v).astype(np.float32)
    return new_p, new_v


def adam_step(params, grads, m, v, t, lr=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-8, l2_reg=0.0):
    """Keras Adam (optimizers.py, decay 0): lr_t = lr*sqrt(1-b2^t)/(1-b1^t); m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
    p -= lr_t * m / (sqrt(v) + eps); kernels get the l2 regulariser's gradient 2*l2*w.  ``t`` counts from 1.  numpy dicts."""
    lr_t = lr * np.sqrt(1.0 - beta_2 ** t) / (1.0 - beta_1 ** t)
    new_p, new_m, new_v = {}, {}, {}
    for k, w in params.items():
        if k not in grads:
            new_p[k] = w
            continue
        g = grads[k].astype(np.float64)
        if k.endswith('/kernel'):
            g = g + 2.0 * l2_reg * w.astype(np.float64)
        mk = beta_1 * m.get(k, 0.0) + (1 - beta_1) * g
        vk = beta_2 * v.get(k, 0.0) + (1 - beta_2) * g * g
        new_m[k], new_v[k] = mk, vk
        new_p[k] = (w.astype(np.float64) - lr_t * mk / (np.sqrt(vk) + epsilon)).astype(np.float32)
    return new_p, new_m, new_v
