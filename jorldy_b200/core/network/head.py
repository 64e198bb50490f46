"""Input heads (jorldy/core/network/head.py): `mlp` = relu(Linear(D_in, H)) (head.py:6-18) and
`cnn` = /255 -> conv 8x8s4 -> 4x4s2 -> 3x3s1 -> flatten (head.py:21-61).

A head owns no storage: it registers its parameter specs on the owning FlatNetwork and runs
forward/backward on that network's flat views.
"""
import torch

from ..dev import C, ptr, stream_ptr
from .base import init_gain, orthogonal_


class MLPHead:
    kind = "mlp"
    max_rows = 16384        # inference chunk: activations (2 x 32 MB at H=512) stay L2-resident
    fwd_launches = 1        # kernels of forward() (launch bookkeeping of the agents and collectors)

    def bwd_launches(self, M):
        return 1

    def __init__(self, D_in, D_hidden=512):
        if not isinstance(D_in, int):
            raise ValueError("mlp head expects an integer state_size")
        self.D_in, self.D_head_out = D_in, D_hidden

    def specs(self):
        return [("head.l.weight", (self.D_head_out, self.D_in)), ("head.l.bias", (self.D_head_out,))]

    def init(self, p, gen=None):
        p["head.l.weight"].copy_(orthogonal_((self.D_head_out, self.D_in), init_gain("relu"), gen))
        p["head.l.bias"].zero_()

    def forward(self, net, x, idx, M, tag, save):
        """x: [rows, D_in] f32 (all rows if idx is None else gathered by idx[M] int32)."""
        h = net._buf(tag + "head.h", (M, self.D_head_out))
        xg = net._buf(tag + "head.xg", (M, self.D_in)) if save else None
        C.jb_mlp_in_fwd(ptr(x), ptr(idx), ptr(net.p["head.l.weight"]), ptr(net.p["head.l.bias"]), M, self.D_in,
                        self.D_head_out, ptr(h), ptr(xg), stream_ptr())
        return h

    def backward(self, net, dh_pre, M, tag):
        """dh_pre: gradient w.r.t. the head's pre-activation (already ReLU-masked)."""
        xg = net._buf(tag + "head.xg", (M, self.D_in))
        C.jb_linear_bwd_dw(ptr(dh_pre), ptr(xg), ptr(net.g["head.l.weight"]), ptr(net.g["head.l.bias"]), M,
                           self.D_in, self.D_head_out, stream_ptr())


class CNNHead:
    """head.py:21-61.  Input: uint8 [rows, C, H, W] (NCHW, as the env / replay produce it)."""
    kind = "cnn"
    max_rows = 256          # inference chunk: the first im2col buffer is 400 KB per row
    fwd_launches = 7        # 3 x (im2col + gemm) + flatten

    def __init__(self, D_in, D_hidden=512):
        C, H, W = D_in
        assert H >= 36 and W >= 36
        self.D_in = (C, H, W)
        self.d1 = ((H - 8) // 4 + 1, (W - 8) // 4 + 1)
        self.d2 = ((self.d1[0] - 4) // 2 + 1, (self.d1[1] - 4) // 2 + 1)
        self.d3 = (self.d2[0] - 3 + 1, self.d2[1] - 3 + 1)
        self.D_head_out = 64 * self.d3[0] * self.d3[1]
        # (name, C_in, C_out, k, stride, in_hw, out_hw)
        self.layers = [("conv1", C, 32, 8, 4, (H, W), self.d1), ("conv2", 32, 64, 4, 2, self.d1, self.d2),
                       ("conv3", 64, 64, 3, 1, self.d2, self.d3)]

    def specs(self):
        out = []
        for name, ci, co, k, s, _, _ in self.layers:
            out += [(f"head.{name}.weight", (co, ci, k, k)), (f"head.{name}.bias", (co,))]
        return out

    def init(self, p, gen=None):
        for name, ci, co, k, s, _, _ in self.layers:
            w = orthogonal_((co, ci * k * k), init_gain("relu"), gen)      # torch flattens dims 1.. the same way
            p[f"head.{name}.weight"].copy_(w.view(co, ci, k, k))
            p[f"head.{name}.bias"].zero_()

    def forward(self, net, x, idx, M, tag, save):
        """x: contiguous uint8 [rows, C, H, W] (all rows if idx is None else gathered by idx[M] int32 inside conv1's
        im2col)."""
        if x.dtype != torch.uint8 or not x.is_contiguous() or tuple(x.shape[1:]) != self.D_in:
            raise ValueError(f"cnn head expects a contiguous uint8 [rows, {', '.join(map(str, self.D_in))}] tensor, "
                             f"got {x.dtype} {tuple(x.shape)}{'' if x.is_contiguous() else ' (non-contiguous)'}")
        if idx is not None and (idx.dtype != torch.int32 or not idx.is_contiguous()):
            raise ValueError(f"cnn head expects contiguous int32 row indices, got {idx.dtype}")
        s = stream_ptr()
        cur = None
        for li, (name, ci, co, k, st, (ih, iw), (oh, ow)) in enumerate(self.layers):
            K = ci * k * k
            col = net._buf(f"{tag}head.col{li}", (M * oh * ow, K))
            if li == 0:
                C.jb_im2col_u8_rows(ptr(x), ptr(idx), M, ci, ih, iw, k, k, st, ptr(col), s)
            else:
                C.jb_im2col_nhwc(ptr(cur), M, ci, ih, iw, k, k, st, ptr(col), s)
            y = net._buf(f"{tag}head.y{li}", (M * oh * ow, co))
            C.jb_linear_fwd(ptr(col), ptr(net.p[f"head.{name}.weight"]), ptr(net.p[f"head.{name}.bias"]), ptr(y),
                            M * oh * ow, K, co, 1, s)
            cur = y
        P = self.d3[0] * self.d3[1]
        feat = net._buf(tag + "head.h", (M, self.D_head_out))
        C.jb_nhwc_to_nchw(ptr(cur), M, P, 64, ptr(feat), s)
        return feat

    def _dw_splits(self, li, M):
        # conv weight gradients are [co, ci k k] = a few 32 x 32 tiles contracted over M * oh * ow rows: split the
        # contraction over the grid (148 SMs) and fold the partials in a fixed order
        _, ci, co, k, _, _, (oh, ow) = self.layers[li]
        tiles = ((ci * k * k + 31) // 32) * ((co + 31) // 32)
        return min(64, max(1, 296 // tiles), max(1, M * oh * ow // 512))

    def bwd_launches(self, M):
        """unflatten + per layer dW (split-K: gemm + 2 folds) + dcol and col2im for conv3 and conv2."""
        return 1 + sum(3 if self._dw_splits(li, M) > 1 else 1 for li in range(3)) + 2 * 2

    def backward(self, net, dfeat_pre, M, tag):
        """dfeat_pre [M, 64*P] (C,H,W order): gradient w.r.t. conv3's pre-activation (already ReLU-masked)."""
        s = stream_ptr()
        P = self.d3[0] * self.d3[1]
        dy = net._buf(tag + "head.dy2", (M * P, 64))
        C.jb_nchw_to_nhwc(ptr(dfeat_pre), M, P, 64, 0, ptr(dy), s)
        for li in (2, 1, 0):
            name, ci, co, k, st, (ih, iw), (oh, ow) = self.layers[li]
            K = ci * k * k
            Mr = M * oh * ow
            col = net._buf(f"{tag}head.col{li}", (Mr, K))
            splits = self._dw_splits(li, M)
            ws = net._buf(f"{tag}head.dwws{li}", (splits * (co * K + co),)) if splits > 1 else None
            C.jb_linear_bwd_dw_splitk(ptr(dy), ptr(col), ptr(net.g[f"head.{name}.weight"]), ptr(net.g[f"head.{name}.bias"]),
                                      Mr, K, co, ptr(ws), splits, s)
            if li == 0:
                break
            dcol = net._buf(f"{tag}head.dcol{li}", (Mr, K))
            C.jb_linear_bwd_dx(ptr(dy), ptr(net.p[f"head.{name}.weight"]), ptr(dcol), Mr, K, co, 0, s)
            y_prev = net._buf(f"{tag}head.y{li - 1}", (M * ih * iw, ci))
            dprev = net._buf(f"{tag}head.dy{li - 1}", (M * ih * iw, ci))
            C.jb_col2im_nhwc(ptr(dcol), M, ci, ih, iw, k, k, st, ptr(y_prev), ptr(dprev), s)
            dy = dprev


head_dict = {"mlp": MLPHead, "cnn": CNNHead}


def make_head(name, D_in, D_hidden):
    if name not in head_dict:
        print(f"### can use only follows {list(head_dict.keys())}")
        raise Exception
    return head_dict[name](D_in, D_hidden)
