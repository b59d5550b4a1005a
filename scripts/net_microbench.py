#!/usr/bin/env python
"""Policy-value forward microbenchmark (GPU): per-layer and whole-forward timing with CUDA
events at the bench batch size.  Not the bench."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rlzero_b200 import _lib as L  # noqa: E402
from rlzero_b200.games.gomoku.policy_value_net import NativeForward, ResNetPolicyValueNet  # noqa: E402


def timeit(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    B = int(os.environ.get('B', 8192))
    blocks = int(os.environ.get('BLOCKS', 10))
    H = int(os.environ.get('H', 15))
    ctas = int(os.environ.get('CTAS', 0))
    torch.manual_seed(0)
    net = ResNetPolicyValueNet(H, n_blocks=blocks).cuda().eval()
    nf = NativeForward(net, max_batch=B, n_ctas=ctas)
    lib = L.load()
    l = nf.layers[1]
    x, y = nf.bufs[0], nf.bufs[1]
    x.normal_()

    flops_alg = 2.0 * B * H * H * 128 * 128 * 9
    flops_issued = 2.0 * B * 256 * 128 * 128 * 9
    z = nf.bufs[1]
    for name, res in (('conv3x3_tc3', None), ('conv3x3_tc3+residual', z)):
        def conv3():
            L.check(lib.rz_net_conv3x3_tc3(L.ptr(x), L.ptr(l['w']), L.ptr(l['b']), L.ptr(res), L.ptr(y), B, H, H,
                                           nf.S, 1, ctas, L.stream_ptr()))
        ms = timeit(conv3)
        print(json.dumps({'kernel': name, 'B': B, 'S': nf.S, 'ms': ms, 'TFLOPs_algorithmic': flops_alg / ms / 1e9,
                          'TFLOPs_issued': 2.0 * B * nf.P * 128 * 128 * 9 / ms / 1e9}))
    if nf.S != 16:
        return
    for name, res in (('conv3x3_tc2', None), ('conv3x3_tc2+residual', z)):
        def conv2():
            L.check(lib.rz_net_conv3x3_tc2(L.ptr(x), L.ptr(l['w']), L.ptr(l['b']), L.ptr(res), L.ptr(y), B, H, H,
                                           128, 1, 2, 0, ctas, L.stream_ptr()))
        ms = timeit(conv2)
        print(json.dumps({'kernel': name, 'B': B, 'ms': ms, 'TFLOPs_algorithmic': flops_alg / ms / 1e9,
                          'TFLOPs_issued': flops_issued / ms / 1e9}))

    def heads_tc():
        L.check(lib.rz_net_heads_tc(nf.hdesc, L.ptr(nf.feat), L.ptr(nf.logp), L.ptr(nf.value), B, L.stream_ptr()))
    print(json.dumps({'kernel': 'heads_tc', 'ms': timeit(heads_tc)}))
    import ctypes as C

    def conv_head():
        L.check(lib.rz_net_conv3x3_tc2_head_ex(L.ptr(x), L.ptr(l['w']), L.ptr(l['b']), L.ptr(z), B, H, H, 128, 1, 0,
                                               nf.w1x1_host.ctypes.data_as(C.c_void_p),
                                               nf.b1x1_host.ctypes.data_as(C.c_void_p), L.ptr(nf.feat), ctas,
                                               L.stream_ptr()))
    ms = timeit(conv_head)
    print(json.dumps({'kernel': 'conv3x3_tc2_head_ex+residual', 'ms': ms, 'TFLOPs_issued': flops_issued / ms / 1e9}))
    rows = torch.zeros(B, 2, H, dtype=torch.int32, device='cuda')
    meta = torch.zeros(B, 12, dtype=torch.int32, device='cuda')
    meta[:, 1] = -1

    g = nf._gdesc()
    st = nf.stem

    def stem():
        L.check(lib.rz_net_stem_tc(C.byref(g), L.ptr(rows), L.ptr(meta), L.ptr(st['w']), L.ptr(st['b']), L.ptr(y), B,
                                   1, 0, L.stream_ptr()))
    print(json.dumps({'kernel': 'stem_fused', 'ms': timeit(stem)}))

    def fwd():
        nf.forward_boards(rows, meta, B)
    ms = timeit(fwd, iters=5, warm=2)
    print(json.dumps({'kernel': 'forward_resnet%d' % blocks, 'B': B, 'ms': ms, 'evals_per_s': B / ms * 1e3,
                      'TFLOPs_algorithmic': net.flops_per_eval() * B / ms / 1e9}))


if __name__ == '__main__':
    main()
