"""Host-side helpers over the C ABI: weight packing, conv descriptors, NHWC buffers."""
from __future__ import annotations

import ctypes as C

import torch

from .. import _lib as L


def pad16(c: int) -> int:
    return (c + 15) // 16 * 16


def fold_bn(w: torch.Tensor, gamma, beta, mean, var, eps: float):
    """Conv(no bias)+BatchNorm -> (w', b').  Same algebra as ultralytics fuse_conv_and_bn (3P) applied by
    model.fuse(); TrackNet's Conv2DBlock (/root/reference/trackers/ball_tracker/models.py:5-17) has the same form."""
    scale = gamma / torch.sqrt(var + eps)
    return w * scale.reshape(-1, 1, 1, 1), beta - mean * scale


def pack_conv_weight(w: torch.Tensor, b: torch.Tensor | None, cin_pad: int, cout_pad: int, device,
                     cin_map: list[int] | None = None):
    """(Cout,Cin,k,k) fp32 -> half [k*k][cout_pad][cin_pad] + float bias [cout_pad] (zero padded).

    cin_map[i] = position of logical input channel i in the padded input tensor (for concat slices that are
    individually padded); default identity."""
    cout, cin, kh, kw = w.shape
    assert kh == kw
    wp = torch.zeros(kh * kw, cout_pad, cin_pad, dtype=torch.float32)
    src = w.detach().float().permute(2, 3, 0, 1).reshape(kh * kw, cout, cin)
    if cin_map is None:
        wp[:, :cout, :cin] = src
    else:
        idx = torch.as_tensor(cin_map, dtype=torch.long)
        wp[:, :cout, idx] = src
    bp = torch.zeros(cout_pad, dtype=torch.float32)
    if b is not None:
        bp[:cout] = b.detach().float()
    return wp.to(torch.float16).contiguous().to(device), bp.contiguous().to(device)


def make_conv_desc(x: torch.Tensor, c_in_off: int, cin: int, w: torch.Tensor, b: torch.Tensor, ksize: int,
                   stride: int, act: int, out: torch.Tensor, out_coff: int, out_mode: int = L.OUT_F16_NHWC,
                   cout_store: int | None = None, res: torch.Tensor | None = None, res_coff: int = 0,
                   head: tuple | None = None, res_before_act: bool = False,
                   out2: tuple | None = None) -> L.ConvDesc:
    """x: NHWC half tensor (N,H,W,C). w: packed half [taps][cout_pad][cin]. out: NHWC tensor (half or float), or
    (N,C,H,W) float for OUT_F32_NCHW. out2 = (NHWC half tensor, first channel, L.OUT2_UP2 | L.OUT2_POOL2): the same
    values written a second time, 2x2-replicated or 2x2-max-pooled (no separate upsample / pool launch)."""
    N, H, W, Ct = x.shape
    cout_pad = w.shape[1]
    assert w.shape[2] == cin and w.shape[0] == ksize * ksize
    d = L.ConvDesc()
    d.in_ = x.data_ptr()
    d.N, d.H, d.W, d.C = N, H, W, Ct
    d.c_in_off, d.cin = c_in_off, cin
    d.weight, d.bias = w.data_ptr(), b.data_ptr()
    d.cout_pad, d.ksize, d.stride, d.act = cout_pad, ksize, stride, act
    d.res_before_act = 1 if res_before_act else 0
    if res is not None:
        d.res, d.res_C, d.res_coff = res.data_ptr(), res.shape[-1], res_coff
    else:
        d.res, d.res_C, d.res_coff = None, 0, 0
    if head is not None:  # (weight float [n][cout_pad], bias float [n], out float (N,n,Ho,Wo))
        hw_, hb_, ho_ = head
        assert hw_.dtype == torch.float32 and hw_.shape[1] == cout_pad and hw_.is_contiguous()
        d.head_weight, d.head_bias, d.head_n, d.head_out = hw_.data_ptr(), hb_.data_ptr(), hw_.shape[0], ho_.data_ptr()
    if out_mode == L.OUT_NONE:
        d.out, d.out_C = None, 0
        d.out_coff, d.out_mode = 0, out_mode
        d.cout_store = cout_pad
        return d
    d.out = out.data_ptr()
    d.out_C = out.shape[-1] if out_mode != L.OUT_F32_NCHW else out.shape[1]
    d.out_coff, d.out_mode = out_coff, out_mode
    d.cout_store = cout_pad if cout_store is None else cout_store
    if out2 is not None:
        t2, off2, mode2 = out2
        Ho, Wo = H // stride, W // stride
        want = (N, 2 * Ho, 2 * Wo) if mode2 == L.OUT2_UP2 else (N, Ho // 2, Wo // 2)
        assert tuple(t2.shape[:3]) == want and t2.dtype == torch.float16, (t2.shape, want)
        d.out2, d.out2_C, d.out2_coff, d.out2_mode = t2.data_ptr(), t2.shape[-1], off2, mode2
    return d


def pack_stem_weight(w: torch.Tensor, b: torch.Tensor | None, cout_pad: int, device):
    """(Cout,3,3,3) fp32 stem weights -> half [3 filter rows][cout_pad][16] with k = s*4 + c (PB_IN_STEM4), + bias."""
    cout = w.shape[0]
    assert tuple(w.shape[1:]) == (3, 3, 3)
    wp = torch.zeros(3, cout_pad, 16, dtype=torch.float32)
    for s in range(3):
        for c in range(3):
            wp[:, :cout, s * 4 + c] = w[:, c, :, s].detach().float().T  # [r][cout]
    bp = torch.zeros(cout_pad, dtype=torch.float32)
    if b is not None:
        bp[:cout] = b.detach().float()
    return wp.to(torch.float16).contiguous().to(device), bp.contiguous().to(device)


def make_stem_desc(x_padded: torch.Tensor, w: torch.Tensor, b: torch.Tensor, act: int, out: torch.Tensor,
                   out_coff: int = 0) -> L.ConvDesc:
    """Stem conv (3x3, stride 2) over the padded 4-channel input (N, H+2, W+2, 4)."""
    N, Hp, Wp, C4 = x_padded.shape
    assert C4 == 4 and w.shape[0] == 3 and w.shape[2] == 16
    d = L.ConvDesc()
    d.in_ = x_padded.data_ptr()
    d.N, d.H, d.W, d.C = N, Hp - 2, Wp - 2, 4
    d.c_in_off, d.cin = 0, 16
    d.weight, d.bias = w.data_ptr(), b.data_ptr()
    d.cout_pad, d.ksize, d.stride, d.act = w.shape[1], 3, 2, act
    d.res, d.res_C, d.res_coff = None, 0, 0
    d.out, d.out_C, d.out_coff, d.out_mode = out.data_ptr(), out.shape[-1], out_coff, L.OUT_F16_NHWC
    d.cout_store = w.shape[1]
    d.in_layout = L.IN_STEM4
    return d


def conv2d(desc: L.ConvDesc, reference: bool = False) -> None:
    fn = L.lib().pb_conv2d_reference if reference else L.lib().pb_conv2d
    L.check(fn(C.byref(desc), L.stream_ptr()))


class Program:
    """Ordered list of device ops bound to fixed buffers (pb_program)."""

    def __init__(self):
        self._h = L.lib().pb_program_create()
        self._keep = []  # tensors referenced by raw pointer
        self.descs: list = []  # per op: ConvDesc copy (convs) or None
        self.kinds: list[str] = []  # per op: 'conv' | 'pool' | 'sppf'
        self.flops: list[float] = []  # per op: algorithmic FLOPs (2*MACs on the real, unpadded channel counts)
        self.bytes: list[float] = []  # per op: algorithmic activation bytes (input read once + output written once)

    def __del__(self):
        try:
            if self._h:
                L.lib().pb_program_destroy(self._h)
        except Exception:
            pass

    def keep(self, *tensors):
        self._keep.extend(tensors)

    def conv(self, desc: L.ConvDesc, cin_real: int | None = None, cout_real: int | None = None):
        L.check(L.lib().pb_program_add_conv(self._h, C.byref(desc)))
        ci = desc.cin if cin_real is None else cin_real
        co = desc.cout_store if cout_real is None else cout_real
        ho, wo = desc.H // desc.stride, desc.W // desc.stride
        self.kinds.append("conv")
        self.descs.append(desc)
        self.flops.append(2.0 * desc.N * ho * wo * co * ci * desc.ksize * desc.ksize)
        obytes = 4 if desc.out_mode in (L.OUT_F32_NHWC, L.OUT_F32_NCHW) else 2
        self.bytes.append(float(desc.N) * (desc.H * desc.W * ci * 2 + ho * wo * co * obytes))

    def maxpool2(self, x, c_off, c, out, out_coff):
        N, H, W, Ct = x.shape
        L.check(L.lib().pb_program_add_maxpool2(self._h, x.data_ptr(), N, H, W, Ct, c_off, c, out.data_ptr(),
                                                out.shape[-1], out_coff))
        self._note("pool", N * H * W * c * 2 * 1.25)

    def sppf_pool(self, buf, c):
        N, H, W, Ct = buf.shape
        L.check(L.lib().pb_program_add_sppf_pool(self._h, buf.data_ptr(), N, H, W, Ct, c))
        self._note("sppf", N * H * W * c * 2 * 4.0)

    def _note(self, kind: str, nbytes: float):
        self.kinds.append(kind)
        self.descs.append(None)
        self.flops.append(0.0)
        self.bytes.append(float(nbytes))

    @property
    def num_ops(self) -> int:
        return L.lib().pb_program_num_ops(self._h)

    def op_kernels(self) -> list[str]:
        names = {0: "conv_tc_kernel", 1: "conv_halo_kernel", 2: "maxpool2_kernel", 4: "sppf_pool_kernel"}
        return [names[L.lib().pb_program_op_kernel(self._h, i)] for i in range(self.num_ops)]

    def run(self, first: int | None = None, last: int | None = None):
        if first is None:
            L.check(L.lib().pb_program_run(self._h, L.stream_ptr()))
        else:
            L.check(L.lib().pb_program_run_range(self._h, first, last, L.stream_ptr()))


def time_program_ops(prog: Program, repeats: int = 5):
    """Per-op device time (ms) with CUDA events recorded on the launch stream between consecutive ops: the MEDIAN of
    `repeats` passes (a best-of-n would flatter the roofline numerator)."""
    import statistics

    n = prog.num_ops
    samples = [[] for _ in range(n)]
    for _ in range(repeats):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        ev[0].record()
        for i in range(n):
            prog.run(i, i + 1)
            ev[i + 1].record()
        torch.cuda.synchronize()
        for i in range(n):
            samples[i].append(ev[i].elapsed_time(ev[i + 1]))
    return [statistics.median(s) for s in samples]
