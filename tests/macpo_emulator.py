"""TEST INFRASTRUCTURE ONLY: torch-CPU emulation of the MACPO entry points of libspo (include/spo.h, csrc/spo_ma_trust.cu) on top of
tests/ma_emulator.EmulatedLib, so that the host orchestration of MACPOTrainer and macpo.Runner runs in the `-m "not gpu"` suite
against the oracle.  Same conventions as ma_emulator: every function takes the C function's positional arguments and "pointers"
are the tensors themselves, treated as flat memory."""
import torch

from ma_emulator import EmulatedLib, _mem, install as _install


class MACPOEmulatedLib(EmulatedLib):
    def spo_ma_ln_in_jvp(self, x, n, K, dw, db, out, stream):
        x = _mem(x, n, K)
        m = x.mean(-1, keepdim=True)
        xh = (x - m) * torch.rsqrt(((x - m) ** 2).mean(-1, keepdim=True) + 1e-5)
        _mem(out, n, K).copy_(xh * _mem(dw, K) + _mem(db, K))
        return 0

    def spo_ma_gemm_nt_pair(self, A1, B1, K1, A2, B2, K2, bias, C, M, N, stream):
        c = _mem(A1, M, K1) @ _mem(B1, N, K1).t() + _mem(A2, M, K2) @ _mem(B2, N, K2).t()
        if bias is not None:
            c = c + _mem(bias, N)
        _mem(C, M, N).copy_(c)
        return 0

    def spo_ma_ln_elu_jvp(self, t, pre, ln_w, dln_w, dln_b, n, H, stream):
        d, e = _mem(t, n, H), _mem(pre, n, H)
        m = e.mean(-1, keepdim=True)
        rstd = torch.rsqrt(((e - m) ** 2).mean(-1, keepdim=True) + 1e-5)
        xh = (e - m) * rstd
        dp = d * torch.where(e > 0, torch.ones_like(e), e + 1)
        y = _mem(ln_w, H) * rstd * (dp - dp.mean(-1, keepdim=True) - xh * (dp * xh).mean(-1, keepdim=True)) + _mem(dln_w, H) * xh + _mem(dln_b, H)
        d.copy_(y)
        return 0

    def spo_ma_fvp_head(self, dmu, n, A, log_std, x_coef, y_coef, dmean, part, stream):
        s = torch.sigmoid(_mem(log_std, A) / x_coef) * y_coef
        dm = _mem(dmu, n, A) * (2.0 / (1e-8 + 2 * s * s)) / n
        _mem(dmean, n, A).copy_(dm)
        nb = (n + 31) // 32
        p = _mem(part, nb, A)
        for blk in range(nb):
            p[blk] = dm[32 * blk:min(n, 32 * blk + 32)].sum(0)
        return 0

    def spo_ma_fvp_finish(self, g, v, count, ls_off, A, log_std, x_coef, y_coef, damping, out, stream):
        g, v, o = _mem(g, count), _mem(v, count), _mem(out, count)
        res = g.clone()
        sg = torch.sigmoid(_mem(log_std, A) / x_coef)
        s = sg * y_coef
        ds = y_coef * sg * (1 - sg) / x_coef
        dds = ds * (1 - 2 * sg) / x_coef
        D = 1e-8 + 2 * s * s
        h = (1 / s ** 2 - 4 * s ** 2 / D ** 2 + 32 * s ** 4 / D ** 3) * ds ** 2 + (-1 / s - 4 * s ** 3 / D ** 2) * dds
        res[ls_off:ls_off + A] = h * v[ls_off:ls_off + A]
        o.copy_(res + damping * v)
        return 0

    def spo_ma_dot(self, x, y, count, part, out, stream):
        _mem(out, 1)[0] = torch.dot(_mem(x, count), _mem(y, count))
        return 0

    def spo_ma_cg_begin(self, b, x, r, p, count, st, part, stream):
        b = _mem(b, count)
        _mem(x, count).zero_()
        _mem(r, count).copy_(b)
        _mem(p, count).copy_(b)
        s = _mem(st, 4)
        s[0], s[1] = torch.dot(b, b), 0.0
        return 0

    def spo_ma_cg_update(self, p, Ap, x, r, count, st, part, tol, stream):
        p, Ap, x, r, s = _mem(p, count), _mem(Ap, count), _mem(x, count), _mem(r, count), _mem(st, 4)
        if s[1] != 0:
            return 0
        alpha = s[0] / (torch.dot(p, Ap) + 1e-8)
        x += alpha * p
        r -= alpha * Ap
        new = torch.dot(r, r)
        p.copy_(r + new / s[0] * p)
        s[0] = new
        if new < tol:
            s[1] = 1.0
        return 0

    def spo_ma_axpby(self, out, a, x, b, y, count, stream):
        res = a * _mem(x, count) + (b * _mem(y, count) if y is not None else 0)
        _mem(out, count).copy_(res)
        return 0

    def spo_ma_clip_norm(self, x, count, max_norm, part, nrm2, stream):
        x = _mem(x, count)
        n2 = torch.dot(x, x)
        _mem(nrm2, 1)[0] = n2
        if torch.sqrt(n2) > max_norm:
            x.copy_(x * max_norm / torch.sqrt(n2))
        return 0

    def spo_ma_linesearch_eval(self, feat, n, H, W, b, log_std, A, actions, old_logp, adv, cost_adv, factor, old_mean, old_std, x_coef, y_coef,
                               part, scalars, stream):
        mu = _mem(feat, n, H) @ _mem(W, A, H).t() + _mem(b, A)
        std = torch.sigmoid(_mem(log_std, A) / x_coef) * y_coef
        lp = -((_mem(actions, n, A) - mu) ** 2) / (2 * std ** 2) - std.log() - 0.9189385332046727
        imp = torch.exp(lp - _mem(old_logp, n, A)).prod(-1)
        so = _mem(old_std, A)
        kl = (so.log() - std.log() + (so ** 2 + (_mem(old_mean, n, A) - mu) ** 2) / (1e-8 + 2 * std ** 2) - 0.5).sum(-1)
        w = imp * _mem(factor, n)
        sc = _mem(scalars, 5)
        sc[0], sc[1], sc[2], sc[3] = -(w * _mem(adv, n)).mean(), (w * _mem(cost_adv, n)).mean(), kl.mean(), imp.mean()
        sc[4] = (0.5 + 0.9189385332046727 + std.log()).mean()
        return 0


def install(monkeypatch):
    lib = _install(monkeypatch)
    from safepo import _lib as L
    mlib = MACPOEmulatedLib()
    monkeypatch.setattr(L, "lib", lambda: mlib)
    return mlib
