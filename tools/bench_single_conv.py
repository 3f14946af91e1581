"""Time mc_conv_fwd alone on given shapes (B C H W O k ...) and report the launch plan it chose."""
import ctypes, json, os, sys, statistics
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import modelcompression_b200 as mc
from modelcompression_b200 import _lib

dev = 'cuda:0'
args = [int(a) for a in sys.argv[1:]]
out = []
for i in range(0, len(args), 6):
    B, C, H, W, O, k = args[i:i + 6]
    conv = mc.MaskedConv2d(C, O, k, 1, (k - 1) // 2, bias=False).to(dev)
    lib = _lib.load()
    LDM = int(os.environ.get('LD_MULT', '8'))
    ld_in, Kc, Npad, ld_out = (C + LDM - 1) // LDM * LDM, (C + (31 if C <= 32 else 63)) // (32 if C <= 32 else 64) * (32 if C <= 32 else 64), (O + 15) // 16 * 16, (O + 7) // 8 * 8
    rows = B * (H + 1) * (W + 1)
    xin = torch.randn(rows, ld_in, device=dev).to(torch.bfloat16)
    wpack = torch.empty(Npad, k * k * Kc, dtype=torch.bfloat16, device=dev)
    scale, shift = torch.ones(Npad, device=dev), torch.zeros(Npad, device=dev)
    yb = torch.empty(rows, ld_out, dtype=torch.bfloat16, device=dev)
    s = _lib.stream_ptr()
    w = conv.weight.data.float().contiguous()
    _lib.check(lib.mc_pack_conv_weights(w.data_ptr(), None, O, C, k, None, O, None, C, wpack.data_ptr(), Npad, Kc, s), "pack")
    d = _lib.mc_conv_desc()
    d.d_in, d.d_wpack, d.d_scale, d.d_shift, d.d_out = xin.data_ptr(), wpack.data_ptr(), scale.data_ptr(), shift.data_ptr(), yb.data_ptr()
    d.B, d.H, d.W, d.Cin, d.Cin_ld, d.N, d.Npad = B, H, W, C, ld_in, O, Npad
    d.ksize, d.leaky, d.epi_mode, d.ldc, d.ch_off, d.block_n, d.stages = k, 1, _lib.MC_EPI_PNHWC, ld_out, 0, 0, 0
    d.block_k = 32 if C <= 32 else 64
    need = int(lib.mc_workspace_bytes_conv_fwd(ctypes.byref(d)))
    if need and not os.environ.get('NO_WS'):
        ws = torch.zeros(need, dtype=torch.uint8, device=dev)
        d.d_ws, d.ws_bytes = ws.data_ptr(), need
    ts = []
    for it in range(12):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            _lib.check(lib.mc_conv_fwd(ctypes.byref(d), s), "conv")
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / 5 * 1e3)
    info = (ctypes.c_int * 8)()
    lib.mc_conv_last_plan(info)
    out.append(dict(ld_in=ld_in, shape=[B, C, H, W, O, k], us=round(statistics.median(ts[2:]), 1), plan=list(info)))
print(json.dumps(out))
