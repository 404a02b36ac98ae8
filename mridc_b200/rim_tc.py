"""Tensor-core time-step engine for RIMBlock (tcgen05 / TMEM kernels of conv_tc.cu and conv_tc2.cu, split-bf16 products).

Used by ``RIMBlock.forward`` when the block has the geometry of the shipped CIRIM/RIM configs
(projects/reconstruction/model_zoo/conf/base_{cirim,rim}_run.yaml, recurrent_layer GRU or IndRNN): two
ConvNonlinear(ReLU) + ConvGRUCell / IndRNNCell (kernel 1) stages with 64 channels and a final 64->2 ConvNonlinear, on images
at least 28 pixels wide (``covers``).  Anything else runs on the generic exact-fp32 CUDA-core kernels.  Both paths are
CUDA; neither is a CPU fallback.

Every activation of the time loop lives in the "BH" layout ([B][H+4][W+4][64 hi bf16 | 64 lo bf16], see conv_tc2.cu): the
hi/lo split is done once by the producing kernel's epilogue, the ConvGRU / IndRNN cells are fed by TMA, and the replicate
padding of ConvNonlinear is the tensor's own border.
"""
import os

import torch

from . import _lib, _ops


def _enabled():
    return os.environ.get("MRIDC_B200_DISABLE_TC", "0") != "1"


_ZERO_STATE = {}
_YH_STATIC = {}      # (B, C, H, W, device) -> [static hybrid k-space buffer, version of the tensor last copied into it]
_GRAPH_POOL = {}     # device -> CUDA-graph memory pool shared by all cascades (they replay one after the other)


def _graphs_enabled(n_px):
    """CUDA-graph replay of a cascade's time loop: MRIDC_B200_GRAPHS=1 always, =0 never; default "auto" = only in the
    launch-bound regime (at most two 320x320 slices per call -- the reference ships batch_size 1,
    base_cirim_run.yaml:71).  Measured on the B200: at 16 slices per call the kernels run back to back anyway (no gain
    device-resident) and a stream of alternating input buffers pays for the captures; at one slice per call the 49
    launches of a cascade cost more than its kernels."""
    v = os.environ.get("MRIDC_B200_GRAPHS", "auto")
    if v == "auto":
        return n_px <= 2 * 320 * 320
    return v != "0"


class RimTcEngine:
    def __init__(self, block):
        from .rim import IndRNNCell

        self.block = block
        self._indrnn = isinstance(block.layers[0].rnn, IndRNNCell)
        self._packs = {}
        self._graphs = {}  # key -> "warm" | (CUDAGraph, static eta, static outputs)

    # ---------------------------------------------------------------------------------------------
    @staticmethod
    def supported(block) -> bool:
        from .rim import ConvGRUCell, ConvNonlinear, IndRNNCell

        if not _enabled() or len(block.layers) != 2 or getattr(block, "conv_dim", 2) != 2:
            return False
        for i, st in enumerate(block.layers):
            c, r = st.convs, st.rnn
            if not isinstance(c, ConvNonlinear) or not isinstance(r, (ConvGRUCell, IndRNNCell)):
                return False
            if type(r) is not type(block.layers[0].rnn):
                return False
            if c._act != _ops.ACT_RELU or c.features != 64 or r.hidden_size != 64 or r.input_size != 64:
                return False
            if r.kernel_size != 1:
                return False
            if i == 0:
                if not (c.input_size == 4 and c.kernel_size == 5 and c.dilation == 1):
                    return False
            else:  # the receptive field of the second conv stays inside the 2-pixel BH border
                if c.input_size != 64 or c.kernel_size % 2 != 1 or c.dilation * (c.kernel_size - 1) // 2 > 2:
                    return False
        f = block.final_layer[0]
        if not isinstance(f, ConvNonlinear) or f.features != 2 or f.input_size != 64 or f._act != _ops.ACT_NONE:
            return False
        return f.kernel_size == 3 and f.dilation == 1

    def covers(self, W) -> bool:
        """The engine runs this block on images W pixels wide: rows of at least 32 positions (W + 4 >= 32), the tile width of
        the BH kernels' loaders and TMA boxes."""
        return self.supported(self.block) and W >= 28

    @staticmethod
    def _g8(lib, B, H, W, dev):
        """Zero-initialised G8 buffer (conv_tc2.cu): the input of the bulk-copy-fed first conv."""
        return torch.zeros(lib.mrb_g8_bytes(B, H, W), dtype=torch.uint8, device=dev)

    def _params(self):
        b = self.block
        ps = []
        for st in b.layers:
            ps += [st.convs.conv_layer.weight, st.rnn.ih.weight, st.rnn.hh if self._indrnn else st.rnn.hh.weight]
        return ps

    def packs(self):
        """Packed (hi/lo split, UMMA-swizzled) weights, rebuilt only when a parameter changes: per layer (conv, cell), the
        first conv has none (mrb_tc2_conv5x5x4 splits its fp32 weights itself)."""
        key = tuple((p.data_ptr(), p._version, str(p.device)) for p in self._params())
        if self._packs.get("key") == key:
            return self._packs["packs"]
        lib = _lib.load()
        st = _lib.stream_ptr()
        b = self.block
        dev = b.layers[0].convs.conv_layer.weight.device
        out = []
        for i, stack in enumerate(b.layers):
            c, r = stack.convs, stack.rnn
            w = c.conv_layer.weight.detach().contiguous()
            pc = None
            if i == 1:
                pc = torch.empty(lib.mrb_tc_packed_floats(0, 64, 64, c.kernel_size), dtype=torch.float32, device=dev)
                _lib.check(lib.mrb_tc_pack_conv(_lib.ptr(w), _lib.ptr(pc), 64, 64, c.kernel_size, st))
            wih = r.ih.weight.detach().contiguous()
            if self._indrnn:  # the 1x1 ih conv; the per-channel recurrent weight goes to the kernel's epilogue
                pg = torch.empty(lib.mrb_tc_packed_floats(0, 64, 64, 1), dtype=torch.float32, device=dev)
                _lib.check(lib.mrb_tc_pack_conv(_lib.ptr(wih), _lib.ptr(pg), 64, 64, 1, st))
            else:  # all 192 gate rows in one CTA (conv_tc2.cu)
                pg = torch.empty(lib.mrb_tc2_gru_packed_bytes(), dtype=torch.uint8, device=dev)
                whh = r.hh.weight.detach().contiguous()
                _lib.check(lib.mrb_tc2_pack_gru(_lib.ptr(wih), _lib.ptr(whh), _lib.ptr(pg), 64, 64, st))
            out.append((pc, pg))
        self._packs.update(key=key, packs=out)
        return out

    def _cell_bh(self, lib, x, h, pack, rnn, h_out, B, H, W, st):
        """ConvGRUCell (rnn_cells.py:93-127) or IndRNNCell (:367-391) with kernel size 1 on BH buffers (conv_tc2.cu:
        gru2_kernel / ind2_kernel)."""
        if self._indrnn:
            _lib.check(lib.mrb_tc2_indrnn(_lib.ptr(x), _lib.ptr(h), _lib.ptr(pack), _lib.ptr(rnn.ih.bias),
                                          _lib.ptr(rnn.hh.detach().reshape(-1)), _lib.ptr(h_out), B, H, W, st))
        else:
            _lib.check(lib.mrb_tc2_gru(_lib.ptr(x), _lib.ptr(h), _lib.ptr(pack), _lib.ptr(rnn.ih.bias), _lib.ptr(h_out),
                                       B, H, W, st))

    # ---------------------------------------------------------------------------------------------
    def conv_stack_bh(self, g4, h, h_alt, xbuf, eta, packs, B, H, W, g8):
        """One time step of the regulariser (rim_block.py:233-248) on BH buffers (conv_tc2.cu): conv5x5 -> ConvGRU -> border
        -> conv3x3(dil) -> ConvGRU -> final conv (tap GEMM) + eta update.  h / h_alt are ping-pong lists, swapped in place."""
        lib = _lib.load()
        st = _lib.stream_ptr()
        b = self.block
        c0, c1 = b.layers[0].convs, b.layers[1].convs
        r0, r1 = b.layers[0].rnn, b.layers[1].rnn
        fin = b.final_layer[0]
        # bulk-copy-fed 5x5: the fp32 gradient is split once into the 16-byte G8 positions, taps are address offsets
        if g4 is not None:  # else: the DC kernel has written g8 itself
            _lib.check(lib.mrb_g8_from_nhwc4(_lib.ptr(g4), _lib.ptr(g8), B, H, W, st))
        _lib.check(lib.mrb_tc2_conv5x5x4(_lib.ptr(g8), _lib.ptr(c0.conv_layer.weight), _lib.ptr(c0.conv_layer.bias),
                                         _lib.ptr(xbuf), B, H, W, 1, st))
        self._cell_bh(lib, xbuf, h[0], packs[0][1], r0, h_alt[0], B, H, W, st)
        h[0], h_alt[0] = h_alt[0], h[0]
        _lib.check(lib.mrb_bh_fix_border(_lib.ptr(h[0]), B, H, W, st))  # the dilated 3x3 reads it spatially
        _lib.check(lib.mrb_tc_conv_bh(_lib.ptr(h[0]), _lib.ptr(packs[1][0]), _lib.ptr(c1.conv_layer.bias), _lib.ptr(xbuf),
                                      B, H, W, 64, c1.kernel_size, c1.dilation, 1, st))
        self._cell_bh(lib, xbuf, h[1], packs[1][1], r1, h_alt[1], B, H, W, st)
        h[1], h_alt[1] = h_alt[1], h[1]
        new_eta = torch.empty_like(eta)
        if B * (H + 4) >= 16:  # the 3-D TMA box of the tap GEMM spans 16 rows of the [B (H+4)] x (W+4) grid
            # tap GEMM on the tensor core + clamped gather: reads the interior of h[1] only, no border fix-up
            _lib.check(lib.mrb_tc2_final_conv(_lib.ptr(h[1]), _lib.ptr(fin.conv_layer.weight), _lib.ptr(fin.conv_layer.bias),
                                              _lib.ptr(eta), _lib.ptr(new_eta), B, H, W, st))
        else:
            _lib.check(lib.mrb_bh_fix_border(_lib.ptr(h[1]), B, H, W, st))  # the CUDA-core 3x3 reads it spatially
            _lib.check(lib.mrb_conv_c2_bh_residual(_lib.ptr(h[1]), _lib.ptr(fin.conv_layer.weight),
                                                   _lib.ptr(fin.conv_layer.bias), _lib.ptr(eta), _lib.ptr(new_eta), B, H, W, st))
        return new_eta

    def bench_step(self, B, H, W, dev):
        """-> (callable running the conv stack of ONE time step on random BH buffers, description)."""
        if not self.covers(W):
            raise ValueError("RimTcEngine.bench_step: the engine does not cover W = %d" % W)
        g4 = torch.randn((B, H, W, 4), device=dev)
        eta = torch.randn((B, H, W, 2), device=dev)
        lib = _lib.load()
        nb = lib.mrb_bh_bytes(B, H, W)
        h, h_alt = [], [torch.empty(nb, dtype=torch.uint8, device=dev) for _ in range(2)]
        for _ in range(2):
            t = torch.randn((B, H, W, 64), device=dev) * 0.1
            buf = torch.empty(nb, dtype=torch.uint8, device=dev)
            _lib.check(lib.mrb_bh_from_nhwc(_lib.ptr(t), _lib.ptr(buf), B, H, W, _lib.stream_ptr()))
            h.append(buf)
        xbuf = torch.empty(nb, dtype=torch.uint8, device=dev)
        packs = self.packs()
        g8 = self._g8(lib, B, H, W, dev)
        if W == 320:
            # production feed at the fastMRI width: the DC kernel writes the G8 conv input itself, so the step starts
            # from a filled G8 buffer (no converter launch)
            _lib.check(lib.mrb_g8_from_nhwc4(_lib.ptr(g4), _lib.ptr(g8), B, H, W, _lib.stream_ptr()))
            g4 = None
        return (lambda: self.conv_stack_bh(g4, h, h_alt, xbuf, eta, packs, B, H, W, g8),
                "split-bf16 tcgen05 ConvGRU stack of one time step on BH activations (bulk-copy-fed conv5x5x4, TMA-fed "
                "ConvGRU, border, conv3x3d2, TMA-fed ConvGRU, tap-GEMM conv3x3->2 + eta)")

    def _steps_bh(self, eta, masked_kspace, sense, mask_can, sigma, h, y_hybrid, ws, fresh_state):
        """The time loop on BH buffers.  h: two BH state buffers (never written); returns (etas, final states)."""
        lib = _lib.load()
        b = self.block
        B, C, H, W, _ = masked_kspace.shape
        dev = masked_kspace.device
        packs = self.packs()
        nb = lib.mrb_bh_bytes(B, H, W)
        h = list(h)
        h_alt = [torch.empty(nb, dtype=torch.uint8, device=dev) for _ in range(2)]
        xbuf = torch.empty(nb, dtype=torch.uint8, device=dev)
        g8 = self._g8(lib, B, H, W, dev)
        # W = 320 row-form DC kernel writes the G8 conv input (split + replicate border) itself: no fp32 gradient tensor
        direct = y_hybrid is not None and W == 320 and C <= 16
        g4 = None if direct else torch.empty((B, H, W, 4), dtype=torch.float32, device=dev)
        etas = []
        for step in range(b.time_steps):
            _ops.dc_rim_grad(eta, masked_kspace, sense, mask_can, sigma, b.fft_centered, b.fft_normalization,
                             out=g8 if direct else g4, ws=ws, nhwc=2 if direct else True, y_hybrid=y_hybrid)
            eta = self.conv_stack_bh(g4, h, h_alt, xbuf, eta, packs, B, H, W, g8)
            if step == 0 and fresh_state:
                # the ping-pong swap left the caller's / the shared zero buffers in h_alt: they must never be written
                h_alt = [torch.empty(nb, dtype=torch.uint8, device=dev) for _ in range(2)]
            etas.append(eta)
        return etas, h

    # ---------------------------------------------------------------------------------------------
    def run(self, eta, masked_kspace, sense, mask_can, sigma, hx, ws, y_hybrid=None, want_hx=True):
        """The time loop of rim_block.py:217-249 on images the engine covers.  eta [B,H,W,2]; hx: list of 2 NCHW-shaped
        tensors or None.  Returns (list of etas, [h0, h1]) with the hidden states NCHW-shaped (channels-last strides);
        ``want_hx=False`` (CIRIM.forward, which drops them, cirim.py:156-163) skips the export of the hidden states."""
        lib = _lib.load()
        b = self.block
        B, C, H, W, _ = masked_kspace.shape
        dev = masked_kspace.device
        st = _lib.stream_ptr()
        nb = lib.mrb_bh_bytes(B, H, W)
        eta = eta.contiguous()
        if hx is None:
            # zero initial state (rim_block.py:188-193): one cached, read-only zero buffer (its border is zero too)
            key = ("bh", B, H, W, str(dev))
            if _ZERO_STATE.get("key") != key:
                _ZERO_STATE.update(key=key, buf=torch.zeros(nb, dtype=torch.uint8, device=dev))
            h = [_ZERO_STATE["buf"], _ZERO_STATE["buf"]]
        else:
            h = []
            for t in hx:  # NCHW fp32 in (the reference API) -> BH; the caller's tensors are never written
                src = _lib.require_cuda(t, "hx").permute(0, 2, 3, 1).contiguous()
                buf = torch.empty(nb, dtype=torch.uint8, device=dev)
                _lib.check(lib.mrb_bh_from_nhwc(_lib.ptr(src), _lib.ptr(buf), B, H, W, st))
                h.append(buf)
        # ---- CUDA-graph replay of the whole time loop (49 launches) when nothing but eta changes between calls: zero initial
        # state, hidden states not wanted (CIRIM.forward), 1-D mask (hybrid k-space), same input tensors as a previous call
        if (hx is None and not want_hx and y_hybrid is not None and _graphs_enabled(B * H * W)
                and not torch.cuda.is_current_stream_capturing()):
            ykey = (B, C, H, W, str(dev))
            ent = _YH_STATIC.get(ykey)
            if ent is None:
                ent = _YH_STATIC[ykey] = [torch.empty_like(y_hybrid), None]
            # once per forward: the cascades share ONE hybrid k-space tensor object, which is marked after the copy.  (An
            # (address, version, id) tag is not enough: the next forward's tensor can reuse all three.)
            if getattr(y_hybrid, "_mrb_static_copy", None) is not ent[0] or y_hybrid._version != ent[1]:
                ent[0].copy_(y_hybrid)
                y_hybrid._mrb_static_copy = ent[0]
                ent[1] = y_hybrid._version
            yh = ent[0]
            pkey = tuple((p.data_ptr(), p._version) for p in self._params())
            gkey = (masked_kspace.data_ptr(), sense.data_ptr(), mask_can.data_ptr(), tuple(masked_kspace.shape),
                    str(mask_can.dtype), tuple(mask_can.shape), float(sigma), bool(b.fft_centered), str(b.fft_normalization),
                    pkey, b.time_steps)
            g = self._graphs.get(gkey)
            if g is None:
                # first sight of these tensors: run eagerly (doubles as the warm-up the capture needs), capture next time
                if len(self._graphs) >= 4:
                    self._graphs.pop(next(iter(self._graphs)))
                self._graphs[gkey] = "warm"
            else:
                if g == "warm":
                    pool = _GRAPH_POOL.get(str(dev))
                    if pool is None:
                        pool = _GRAPH_POOL[str(dev)] = torch.cuda.graph_pool_handle()
                    graph = torch.cuda.CUDAGraph()
                    eta_in = eta.clone()
                    n0 = _lib.launch_count()
                    with torch.cuda.graph(graph, pool=pool):
                        outs, _ = self._steps_bh(eta_in, masked_kspace, sense, mask_can, sigma, h, yh, ws, True)
                        outs = torch.stack(outs)
                    n_launch = _lib.launch_count() - n0  # launches of this library inside the graph
                    lib.mrb_add_launch_count(-n_launch)   # captured, not executed
                    # the tuple keeps every tensor the graph reads alive
                    g = self._graphs[gkey] = (graph, eta_in, outs, n_launch, (masked_kspace, sense, mask_can, yh, h))
                graph, eta_in, outs, n_launch = g[0], g[1], g[2], g[3]
                eta_in.copy_(eta)
                graph.replay()
                lib.mrb_add_launch_count(n_launch)
                return list(outs.clone().unbind(0)), None  # the static outputs are overwritten by the next replay
        etas, h = self._steps_bh(eta, masked_kspace, sense, mask_can, sigma, h, y_hybrid, ws, True)
        if not want_hx:
            return etas, None
        out = []
        for buf in h:  # BH -> fp32, NCHW-shaped like the reference's hidden states
            t = torch.empty((B, H, W, 64), dtype=torch.float32, device=dev)
            _lib.check(lib.mrb_bh_to_nhwc(_lib.ptr(buf), _lib.ptr(t), B, H, W, st))
            out.append(t.permute(0, 3, 1, 2))
        return etas, out

