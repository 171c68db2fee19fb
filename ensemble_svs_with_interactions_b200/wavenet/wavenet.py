"""WaveNet — drop-in for ``nnsvs.wavenet.WaveNet`` (nnsvs/wavenet/wavenet.py:7-171)."""
import torch
from torch import nn
from torch.nn import functional as F

from .. import _lib as _L
from .. import ops
from .modules import Conv1d1x1, ResSkipBlock
from .training import _dims, _forward, _pack, _params, wavenet_forward_with_grad

f32 = torch.float32


def _weights(net):
    """training._params, detached: the parameters stacked over the layers, as the inference packs read them."""
    return {k: None if t is None else t.detach() for k, t in _params(net)}


class WaveNet(nn.Module):
    def __init__(self, in_dim=334, out_dim=206, layers=10, stacks=1, residual_channels=64, gate_channels=128,
                 skip_out_channels=64, kernel_size=3):
        super().__init__()
        self.in_dim = in_dim
        self.out_dim = out_dim
        self.first_conv = Conv1d1x1(out_dim, residual_channels)
        self.main_conv_layers = nn.ModuleList()
        layers_per_stack = layers // stacks
        for layer in range(layers):
            self.main_conv_layers.append(ResSkipBlock(residual_channels, gate_channels, kernel_size, skip_out_channels,
                                                      dilation=2 ** (layer % layers_per_stack), cin_channels=in_dim))
        self.last_conv_layers = nn.ModuleList([nn.ReLU(), Conv1d1x1(skip_out_channels, skip_out_channels), nn.ReLU(),
                                               Conv1d1x1(skip_out_channels, out_dim)])
        self.use_cuda_graph = True

    def _packed(self):
        """(sizes, dilations, weight pack, stacked parameters) of the inference forward, rebuilt when any parameter
        changes: the leading arguments of training._forward."""
        key = tuple((q.data_ptr(), q._version) for q in self.parameters())
        if self.__dict__.get("_pack_key") != key:
            (dims, dilations), w = _dims(self), _weights(self)
            self.__dict__["_pack"] = (dims, dilations, _pack(dims, w), w)
            self.__dict__["_pack_key"] = key
        return self.__dict__["_pack"]

    def forward(self, c, x, lengths=None):
        """c (B,T,in_dim) conditioning, x (B,T,out_dim) targets -> (B,T,out_dim)   (wavenet.py:60-87).

        Differentiable only in training mode: when the module is in training mode, grad mode is on and c, x or a
        parameter requires grad, the output has a grad_fn and ``backward()`` fills the gradients of the parameters
        (weight_g / weight_v, or weight after remove_weight_norm_(), and the biases) and of c / x on libsvsk kernels
        (wavenet/training.py).  Every other call, eval mode included even with grad mode on, runs the inference path
        below and returns a tensor without grad_fn; that differs from a plain nn.Module, which records gradients in
        eval mode too.  Both paths compute the same output bits."""
        if self.training and torch.is_grad_enabled() and (
                c.requires_grad or x.requires_grad or any(q.requires_grad for q in self.parameters())):
            return wavenet_forward_with_grad(self, c, x)
        return self._forward_no_grad(c, x)

    @torch.no_grad()
    def _forward_no_grad(self, c, x):
        """The inference path of forward.  The network is launch-latency bound (138 MFLOP at the reference test's
        shape): the second call of a shape captures the launches as one CUDA graph, later calls replay it.  The kernels
        are training._forward's (svsk_wavenet_block_f32 for the blocks) on a pack built once per parameter version."""
        if not x.is_cuda:
            raise RuntimeError("WaveNet runs on CUDA (sm_100a) only: libsvsk has no CPU path")
        x = x.to(f32).transpose(1, 2).contiguous()
        c = c.to(f32).transpose(1, 2).contiguous()
        plist = self.__dict__.get("_plist")           # walking the module tree costs more than the 5 launches of a forward
        if plist is None:
            plist = self.__dict__["_plist"] = list(self.parameters())
        key = (tuple(c.shape), tuple(x.shape), plist[0].data_ptr(), tuple(q._version for q in plist))
        ent = self.__dict__.setdefault("_graphs", {}).get(key)
        if ent is None and self.use_cuda_graph and not torch.cuda.is_current_stream_capturing():
            seen = self.__dict__.setdefault("_seen", {})
            seen[key] = seen.get(key, 0) + 1
            if seen[key] >= 2:
                if len(self._graphs) >= 4:
                    self._graphs.clear()
                seen.clear()
                s_c, s_x = c.clone(), x.clone()
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):           # warm-up outside capture: the weight pack, allocator pools
                    _forward(*self._packed(), s_c, s_x, train=False)
                torch.cuda.current_stream().wait_stream(side)
                g = torch.cuda.CUDAGraph()
                n0 = _L.launch_count
                with torch.cuda.graph(g):
                    out = _forward(*self._packed(), s_c, s_x, train=False)[0]
                ent = self._graphs[key] = (g, s_c, s_x, out, _L.launch_count - n0)
                _L.launch_count = n0
        if ent is None:
            return _forward(*self._packed(), c, x, train=False)[0].transpose(1, 2)
        g, s_c, s_x, out, n = ent
        s_c.copy_(c); s_x.copy_(x)
        g.replay()
        _L.launch_count += n
        return out.clone().transpose(1, 2)

    def _ar_config(self):
        """(out_dim, R, G, S, layers, stacks, ksize) when svsk_wavenet_ar_f32 covers this network, else None."""
        blocks = self.main_conv_layers
        L = len(blocks)
        dil = [f.dilation for f in blocks]
        per = dil.index(1, 1) if 1 in dil[1:] else L
        if L % per or dil != [2 ** (i % per) for i in range(L)] or len({f.kernel_size for f in blocks}) != 1:
            return None
        cfg = (self.out_dim, self.first_conv.out_channels, blocks[0].conv.out_channels, blocks[0].conv1x1_skip.out_channels,
               L, L // per, blocks[0].kernel_size)
        return cfg if ops.wavenet_ar_supported(*cfg) else None

    def _ar_packed(self, cfg):
        """Folded, laid-out weights of the device sampler, rebuilt when any parameter changes."""
        key = (cfg,) + tuple((q.data_ptr(), q._version) for q in self.parameters())
        if self.__dict__.get("_ar_key") != key:
            out_dim, R, G, S, layers, stacks, k = cfg
            self.__dict__["_ar_pack"] = ops.wavenet_ar_pack_f32(
                _weights(self), out_dim=out_dim, R=R, G=G, S=S, cin=self.main_conv_layers[0].conv1x1c.in_channels,
                layers=layers, stacks=stacks, ksize=k)
            self.__dict__["_ar_key"] = key
        return self.__dict__["_ar_pack"]

    @torch.no_grad()
    def inference(self, c, num_time_steps=100, tqdm=lambda x: x, *, u=None, logits=None):
        """Autoregressive sampling (wavenet.py:89-149): c (B, T >= num_time_steps, in_dim) -> one-hot samples
        (B, num_time_steps, out_dim).

        On CUDA in eval mode, for the shapes svsk_wavenet_ar_supported covers, all steps run in one launch
        (svsk_wavenet_ar_f32, after one svsk_conv1d_f32 for the conditioning of every layer); ``tqdm`` is not used there.
        Step t draws the smallest class whose cumulative softmax probability exceeds u[b, t]: ``u`` (B, num_time_steps)
        fp32 uniforms in [0, 1) is drawn with torch.rand unless given; ``logits`` (B, num_time_steps, out_dim) fp32, if
        given, receives the logits of every step.  Other inputs run the per-step host loop of the reference (per-layer
        ring buffers, OneHotCategorical), which takes neither ``u`` nor ``logits``."""
        cfg = self._ar_config() if c.is_cuda and not self.training else None
        if cfg is not None:
            out_dim, R, G, S, layers, stacks, k = cfg
            self.clear_buffer()
            wpack, wcond = self._ar_packed(cfg)
            cproj = ops.conv1d_f32(c[:, :num_time_steps].to(f32).transpose(1, 2).contiguous(), wcond)
            if u is None:
                u = torch.rand((c.shape[0], num_time_steps), device=c.device)
            y = ops.wavenet_ar_f32(wpack, cproj, u, out_dim=out_dim, R=R, G=G, S=S, layers=layers, stacks=stacks, ksize=k,
                                   logits=logits)
            self.clear_buffer()
            return y
        if u is not None or logits is not None:
            raise ValueError("WaveNet.inference: u= and logits= need the device sampler (CUDA tensors, eval mode, a shape "
                             "svsk_wavenet_ar_supported covers)")
        self.clear_buffer()
        B = c.shape[0]
        outputs = []
        current = torch.zeros(B, 1, self.out_dim, device=c.device)
        steps = range(num_time_steps) if tqdm is None else tqdm(range(num_time_steps))
        for t in steps:
            if t > 0:
                current = outputs[-1]
            x = self.incremental_logits(current, c[:, t, :].unsqueeze(1))
            probs = F.softmax(x.view(B, -1), dim=1)
            outputs.append(torch.distributions.OneHotCategorical(probs).sample().view(B, 1, -1))
        out = torch.cat(outputs, dim=1)
        self.clear_buffer()
        return out

    @torch.no_grad()
    def incremental_logits(self, current, ct):
        """One step of the incremental network (wavenet.py:117-139): current (B,1,out_dim) = the previous frame's
        output (zeros at t = 0), ct (B,1,in_dim) -> logits (B,1,out_dim); the per-layer ring buffers advance by one."""
        x = self.first_conv.incremental_forward(current)
        skips = 0
        for f in self.main_conv_layers:
            x, h = f.incremental_forward(x, ct)
            skips = skips + h
        x = skips
        for f in self.last_conv_layers:
            x = f.incremental_forward(x) if hasattr(f, "incremental_forward") else f(x)
        return x

    def clear_buffer(self):
        self.first_conv.clear_buffer()
        for f in self.main_conv_layers:
            f.clear_buffer()
        for f in self.last_conv_layers:
            if hasattr(f, "clear_buffer"):
                f.clear_buffer()

    def remove_weight_norm_(self):
        def _remove(m):
            try:
                torch.nn.utils.remove_weight_norm(m)
            except ValueError:
                return

        self.apply(_remove)
        self.__dict__.pop("_plist", None)     # the parameters were replaced
        self.__dict__.pop("_graphs", None)
