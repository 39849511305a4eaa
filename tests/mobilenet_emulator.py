"""CPU (torch fp32) interpreter of the op list that openpifpaf_b200.network.build_ops emits for a MobileNet plan.

Test infrastructure, the MobileNet counterpart of tests/ops_emulator.py: it executes the ops exactly as the C ABI
documents them (include/pifpaf_b200.h), with the activation codes (0 none, 1 ReLU, 2 ReLU6, 3 Hardswish) and the
'se_conv1x1' op (squeeze-excitation folded into per-image projection weights).  bf16=True rounds to bf16 where the
kernels do: activations after every op and the GEMM weights (the depthwise kernel k_dwconv_nc keeps f32 weights)."""
import torch
import torch.nn.functional as F


def _act(y, code):
    if code == 1:
        return F.relu(y)
    if code == 2:
        return F.relu6(y)
    if code == 3:
        return F.hardswish(y)
    return y


def run_ops(tensors, ops, images, bf16=False):
    """images [B,3,H,W] float32 -> (list of head outputs [B,F,comp,h,w], activation tensors [B,h,w,c_phys])"""
    B = images.shape[0]
    acts = [torch.zeros((B, h, w, c), dtype=torch.float32) for (h, w, c) in tensors]

    def q(x):
        return x.to(torch.bfloat16).to(torch.float32) if bf16 else x

    heads_out = None
    for o in ops:
        kind = o['kind']
        if kind == 'input_conv':
            y = F.conv2d(images, torch.from_numpy(o['w']), torch.from_numpy(o['b']), o['stride'], o['pad'])
            acts[o['out']][..., :o['c_out']] = q(_act(y, o['relu']).permute(0, 2, 3, 1))
        elif kind == 'conv1x1':
            assert o['shuffle_src'] < 0 and 'pieces' not in o
            a = acts[o['in']][..., o['in_off']:o['in_off'] + o['k_cols']]
            y = _act(a @ q(torch.from_numpy(o['w'])).t() + torch.from_numpy(o['b']), o['relu'])
            acts[o['out']][..., o['out_off']:o['out_off'] + o['n_out']] = q(y)
        elif kind == 'conv':
            a = acts[o['in']][..., o['in_off']:o['in_off'] + o['c_in']].permute(0, 3, 1, 2)
            y = F.conv2d(a, q(torch.from_numpy(o['w'])), torch.from_numpy(o['b']), o['stride'], o['pad'])
            y = y.permute(0, 2, 3, 1)
            if o['residual'] >= 0:
                y = y + acts[o['residual']][..., o['residual_off']:o['residual_off'] + o['n_out']]
            acts[o['out']][..., o['out_off']:o['out_off'] + o['n_out']] = q(_act(y, o['relu']))
        elif kind == 'dwconv':
            c = o['channels']
            a = acts[o['in']][..., o['in_off']:o['in_off'] + c].permute(0, 3, 1, 2)
            w = torch.from_numpy(o['w']).reshape(c, 1, o['kernel'], o['kernel'])
            y = F.conv2d(a, w, torch.from_numpy(o['b']), o['stride'], o['pad'], groups=c)
            acts[o['out']][..., o['out_off']:o['out_off'] + c] = q(_act(y, o['relu']).permute(0, 2, 3, 1))
        elif kind == 'se_conv1x1':
            # SqueezeExcitation (avg-pool, fc1, ReLU, fc2, Hardsigmoid) folded into per-image projection weights
            # bf16(W * s[b]); then the linear projection (+ residual)
            c, n = o['channels'], o['n_out']
            x = acts[o['in']][..., :c]
            pooled = x.mean(dim=(1, 2))
            hid = F.relu(pooled @ torch.from_numpy(o['fc1_w']).t() + torch.from_numpy(o['fc1_b']))
            s = F.hardsigmoid(hid @ torch.from_numpy(o['fc2_w']).t() + torch.from_numpy(o['fc2_b']))
            w = q(torch.from_numpy(o['w'])[None] * s[:, None, :])                   # [B, n, c]
            y = torch.einsum('bhwc,bnc->bhwn', x, w) + torch.from_numpy(o['b'])
            if o['residual'] >= 0:
                y = y + acts[o['residual']][..., :n]
            acts[o['out']][..., :n] = q(y)
        elif kind == 'heads':
            a = acts[o['in']][..., :o['k_cols']]
            y = a @ q(torch.from_numpy(o['w'])).t() + torch.from_numpy(o['b'])   # [B,h,w,N]
            _, h, w, _ = y.shape
            xs = torch.arange(w, dtype=torch.float32).view(1, 1, w)
            ys = torch.arange(h, dtype=torch.float32).view(1, h, 1)
            heads_out, col, op_off = [], 0, 0
            for nf, nc in zip(o['n_fields'], o['n_comp']):
                t = y[..., col:col + nf * nc].reshape(B, h, w, nf, nc).permute(0, 3, 4, 1, 2).clone()
                for c_i in range(nc):
                    op = o['ops'][op_off + c_i]
                    if op == 1:
                        t[:, :, c_i] = torch.sigmoid(t[:, :, c_i])
                    elif op == 2:
                        t[:, :, c_i] += xs
                    elif op == 3:
                        t[:, :, c_i] += ys
                    elif op == 4:
                        t[:, :, c_i] = F.softplus(t[:, :, c_i])
                heads_out.append(t)
                col += nf * nc
                op_off += nc
        else:
            raise ValueError(kind)
    return heads_out, acts
