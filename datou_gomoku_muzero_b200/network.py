"""GomokuNetEZ-compatible network (reference network.py:109-152): representation / prediction /
dynamics towers with the same parameter names, so a reference `state_dict` loads unchanged.

The conv stack is the one dense contraction on the path and stays in PyTorch (cuDNN / cuBLAS
tensor-core kernels) -- SURVEY section 2 row 4 "called, not rewritten".  What this module adds for the
engine is `DeviceEvaluator`: the network frozen for inference (eval BatchNorm, bf16, channels_last,
optionally CUDA-graph captured at the engine's batch size) as a callable
`obs f32 [G,3,N,N] -> (logits f32 [G,A], values f32 [G])` with no host round trip.
"""
from __future__ import annotations

import copy

import torch
import torch.nn as nn
import torch.nn.functional as F


def capture_stream(device):
    """The stream to capture a searcher's step graph on: the current one (the stream of the engine being driven), unless
    that is the legacy default stream, which cannot be captured (torch.cuda.graph then uses its own side stream)."""
    cur = torch.cuda.current_stream(device)
    return None if cur == torch.cuda.default_stream(device) else cur


def _c3(cin, cout):
    return nn.Conv2d(cin, cout, 3, padding=1, bias=False)


class _Res(nn.Module):
    """conv-bn-relu-conv-bn + skip, relu (EvarResBlock, network.py:30-47); bn2 gain starts at 0."""

    def __init__(self, ch):
        super().__init__()
        self.conv1, self.bn1 = _c3(ch, ch), nn.BatchNorm2d(ch, eps=1e-4)
        self.conv2, self.bn2 = _c3(ch, ch), nn.BatchNorm2d(ch, eps=1e-4)
        nn.init.constant_(self.bn2.weight, 0)

    def forward(self, x):
        y = F.relu(self.bn1(self.conv1(x)))
        return F.relu(self.bn2(self.conv2(y)) + x)


class _Representation(nn.Module):
    def __init__(self, planes, blocks, ch):
        super().__init__()
        self.conv, self.bn = _c3(planes, ch), nn.BatchNorm2d(ch, eps=1e-4)
        self.resblocks = nn.Sequential(*[_Res(ch) for _ in range(blocks)])

    def forward(self, x):
        return self.resblocks(F.relu(self.bn(self.conv(x))))


class _Prediction(nn.Module):
    def __init__(self, ch, n, actions, bins, hidden):
        super().__init__()
        self.policy_conv, self.policy_bn = nn.Conv2d(ch, 2, 1), nn.BatchNorm2d(2, eps=1e-4)
        self.policy_fc = nn.Linear(2 * n * n, actions)
        self.value_conv, self.value_bn = nn.Conv2d(ch, 1, 1), nn.BatchNorm2d(1, eps=1e-4)
        self.value_fc1, self.value_fc2 = nn.Linear(n * n, hidden), nn.Linear(hidden, bins)

    def forward(self, h):
        b = h.size(0)
        p = F.relu(self.policy_bn(self.policy_conv(h))).reshape(b, -1)
        v = F.relu(self.value_bn(self.value_conv(h))).reshape(b, -1)
        return self.policy_fc(p), self.value_fc2(F.relu(self.value_fc1(v)))


class _Dynamics(nn.Module):
    def __init__(self, ch, n, bins, hidden, blocks, embed=16):
        super().__init__()
        self.action_embed_conv = nn.Conv2d(1, embed, 1, bias=False)
        self.conv, self.bn = _c3(ch + embed, ch), nn.BatchNorm2d(ch, eps=1e-4)
        self.resblocks = nn.Sequential(*[_Res(ch) for _ in range(blocks)])
        self.reward_fc = nn.Sequential(nn.Linear(ch * n * n, hidden), nn.ReLU(), nn.Linear(hidden, bins))

    def forward(self, state, action):
        b, _, n, m = state.shape
        plane = F.one_hot(action.reshape(b), n * m).to(state.dtype).reshape(b, 1, n, m)
        x = torch.cat((state, self.action_embed_conv(plane)), dim=1)
        nxt = self.resblocks(F.relu(self.bn(self.conv(x))))
        return nxt, self.reward_fc(nxt.reshape(b, -1))


class _Projection(nn.Module):
    def __init__(self, dim, hidden=512, out=512):
        super().__init__()
        self.fc1, self.bn1, self.fc2 = nn.Linear(dim, hidden), nn.BatchNorm1d(hidden, eps=1e-4), nn.Linear(hidden, out)

    def forward(self, x):
        return self.fc2(F.relu(self.bn1(self.fc1(x.reshape(x.size(0), -1)))))


def _support_scalar(logits, lo, hi, bins):
    """softmax over the support bins dotted with linspace(lo, hi, bins) (network.py:9-13)."""
    support = torch.linspace(lo, hi, bins, device=logits.device, dtype=logits.dtype)
    return (F.softmax(logits, dim=1) * support).sum(dim=1, keepdim=True)


class GomokuNetEZ(nn.Module):
    def __init__(self, config_obj):
        super().__init__()
        c = config_obj
        n, ch, blocks, hid = c.BOARD_SIZE, c.NUM_FILTERS, c.NUM_RES_BLOCKS, c.HEAD_HIDDEN_DIM
        self.board_size, self.action_space_size = n, c.ACTION_SPACE_SIZE
        self.v_sup = (c.VALUE_SUPPORT_MIN, c.VALUE_SUPPORT_MAX, c.VALUE_SUPPORT_BINS)
        self.r_sup = (c.REWARD_SUPPORT_MIN, c.REWARD_SUPPORT_MAX, c.REWARD_SUPPORT_BINS)
        self.representation_net = _Representation(3, blocks, ch)
        self.prediction_net = _Prediction(ch, n, self.action_space_size, self.v_sup[2], hid)
        self.dynamics_net = _Dynamics(ch, n, self.r_sup[2], hid, blocks)
        self.projection_net = _Projection(ch * n * n)

    def representation(self, obs):
        return self.representation_net(obs)

    def prediction(self, hidden):
        return self.prediction_net(hidden)

    def dynamics(self, hidden, action):
        return self.dynamics_net(hidden, action.squeeze(-1))

    def project(self, hidden, with_grad=True):
        if with_grad:
            return self.projection_net(hidden)
        with torch.no_grad():
            return self.projection_net(hidden)

    @torch.no_grad()
    def initial_inference(self, obs):
        self.eval()
        hidden = self.representation(obs)
        policy_logits, value_logits = self.prediction(hidden)
        return policy_logits, _support_scalar(value_logits, *self.v_sup), hidden

    @torch.no_grad()
    def recurrent_inference(self, hidden, action):
        self.eval()
        nxt, reward_logits = self.dynamics(hidden, action)
        policy_logits, value_logits = self.prediction(nxt)
        return (policy_logits, _support_scalar(value_logits, *self.v_sup), nxt,
                _support_scalar(reward_logits, *self.r_sup))


def _fold(conv: nn.Conv2d, bn: nn.BatchNorm2d, dtype):
    """Eval-mode BatchNorm folded into the preceding conv: (W', b') with bn(conv(x)) == conv'(x)."""
    scale = bn.weight.float() / torch.sqrt(bn.running_var.float() + bn.eps)
    w = conv.weight.float() * scale.reshape(-1, 1, 1, 1)
    b = bn.bias.float() - bn.running_mean.float() * scale
    if conv.bias is not None:
        b = b + conv.bias.float() * scale
    return (w.to(dtype).contiguous(memory_format=torch.channels_last), b.to(dtype).contiguous())


def _fold_heads(p, dtype):
    """The two 1x1 head convs (policy: 2 channels, value: 1 channel; network.py:50-58 of the reference
    layout) as ONE 3-channel conv, so the hidden state is read once.  A 1-channel conv on its own is
    dispatched to a GEMV kernel that runs at a fifth of the HBM rate."""
    (wp, bp), (wv, bv) = _fold(p.policy_conv, p.policy_bn, dtype), _fold(p.value_conv, p.value_bn, dtype)
    return torch.cat((wp, wv), 0).contiguous(memory_format=torch.channels_last), torch.cat((bp, bv), 0).contiguous()


class FoldedInitialInference:
    """`initial_inference` (network.py:137-143) with every BatchNorm folded into its conv and the
    conv + bias + (residual) + ReLU groups issued as single cuDNN fused ops
    (`cudnn_convolution_relu` / `cudnn_convolution_add_relu`): ~3x fewer kernels and no separate
    elementwise passes over the [B,128,N,N] activations.  Library kernels, inference only."""

    def __init__(self, net: "GomokuNetEZ", dtype=torch.bfloat16):
        self.dtype = dtype
        r, p = net.representation_net, net.prediction_net
        self.stem = _fold(r.conv, r.bn, dtype)
        self.blocks = [(_fold(b.conv1, b.bn1, dtype), _fold(b.conv2, b.bn2, dtype)) for b in r.resblocks]
        self.pv = _fold_heads(p, dtype)
        self.policy_fc = (p.policy_fc.weight.to(dtype), p.policy_fc.bias.to(dtype))
        self.value_fc1 = (p.value_fc1.weight.to(dtype), p.value_fc1.bias.to(dtype))
        self.value_fc2 = (p.value_fc2.weight.to(dtype), p.value_fc2.bias.to(dtype))
        self.v_sup = net.v_sup
        self.fused = True

    def _conv_relu(self, x, wb, pad):
        w, b = wb
        if self.fused:
            return torch.cudnn_convolution_relu(x, w, b, (1, 1), (pad, pad), (1, 1), 1)
        return F.relu(F.conv2d(x, w, b, padding=pad))

    def _conv_add_relu(self, x, wb, z):
        w, b = wb
        if self.fused:
            return torch.cudnn_convolution_add_relu(x, w, z, 1.0, b, (1, 1), (1, 1), (1, 1), 1)
        return F.relu(F.conv2d(x, w, b, padding=1) + z)

    @torch.no_grad()
    def __call__(self, x):
        h = self._conv_relu(x, self.stem, 1)
        for c1, c2 in self.blocks:
            h = self._conv_add_relu(self._conv_relu(h, c1, 1), c2, h)
        b = h.size(0)
        pv = self._conv_relu(h, self.pv, 0)
        pl, vl = pv[:, :2].reshape(b, -1), pv[:, 2].reshape(b, -1)
        logits = F.linear(pl, *self.policy_fc)
        vlog = F.linear(F.relu(F.linear(vl, *self.value_fc1)), *self.value_fc2)
        return logits, _support_scalar(vlog.float(), *self.v_sup), h


class DeviceEvaluator:
    """`initial_inference` frozen for the engine: obs f32 [B,3,N,N] (engine-owned, fixed address) ->
    (logits f32 [B,A], values f32 [B]) written into fixed output buffers.  bf16 + channels_last by
    default; with `graph=True` the forward is captured once in a CUDA graph and replayed, so a
    simulation step is {select kernel, one graph launch, expand/backup kernel}."""

    def __init__(self, net: GomokuNetEZ, obs_buffer: torch.Tensor, dtype=torch.bfloat16, graph=True, folded=True):
        torch.backends.cudnn.benchmark = True      # let cuDNN pick the conv algorithm for this fixed shape
        self.net = copy.deepcopy(net).to(obs_buffer.device).eval()    # the caller's module is left untouched
        self.dtype = dtype
        self.folded = FoldedInitialInference(self.net, dtype) if folded else None
        if dtype != torch.float32:
            self.net = self.net.to(dtype)
        self.net = self.net.to(memory_format=torch.channels_last)
        self.obs = obs_buffer
        if self.folded is not None:
            try:        # the fused cuDNN entry points do not cover every dtype / build
                self.folded(obs_buffer[:2].to(dtype).contiguous(memory_format=torch.channels_last))
            except RuntimeError:
                self.folded.fused = False
        B = obs_buffer.shape[0]
        self.logits = torch.empty((B, net.action_space_size), dtype=torch.float32, device=obs_buffer.device)
        self.values = torch.empty(B, dtype=torch.float32, device=obs_buffer.device)
        self.graph = None
        if graph:
            s = torch.cuda.Stream(device=obs_buffer.device)
            s.wait_stream(torch.cuda.current_stream(obs_buffer.device))
            with torch.cuda.stream(s):
                for _ in range(3):
                    self._forward()
            torch.cuda.current_stream(obs_buffer.device).wait_stream(s)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._forward()

    @torch.no_grad()
    def _forward(self):
        x = self.obs                 # already the network's input format when the select wrote bf16 NHWC: no cast, no re-layout
        if x.dtype != self.dtype or not x.is_contiguous(memory_format=torch.channels_last):
            x = x.to(self.dtype).contiguous(memory_format=torch.channels_last)
        p, v, _ = self.folded(x) if self.folded is not None else self.net.initial_inference(x)
        self.logits.copy_(p)
        self.values.copy_(v.reshape(-1))

    def update_weights(self, state_dict):
        """Hot-swap the evaluator's weights (the reference's ModelWeightsUpdate message,
        workers.py:331-335, ipc_messages.py:75-77): load the full state_dict and refold IN PLACE,
        so a captured CUDA graph keeps replaying against the same buffers.  Folding starts from an fp32
        copy of the new weights -- exactly what __init__ does -- so update_weights(sd) gives the same folded
        tensors as DeviceEvaluator(net_with_sd) (no double rounding through the inference dtype)."""
        master = copy.deepcopy(self.net).float()
        master.load_state_dict({k: v.float() if v.is_floating_point() else v for k, v in state_dict.items()})
        self.net.load_state_dict({k: v.to(self.dtype) if v.is_floating_point() else v for k, v in master.state_dict().items()})
        if self.folded is not None:
            fresh = FoldedInitialInference(master.to(self.obs.device).eval(), self.dtype)
            old, new = self.folded, fresh
            with torch.no_grad():
                for a, b in zip([old.stem, *sum(([x, y] for x, y in old.blocks), []), old.pv,
                                 old.policy_fc, old.value_fc1, old.value_fc2],
                                [new.stem, *sum(([x, y] for x, y in new.blocks), []), new.pv,
                                 new.policy_fc, new.value_fc1, new.value_fc2]):
                    a[0].copy_(b[0]); a[1].copy_(b[1])

    def __call__(self, obs):
        if obs.data_ptr() != self.obs.data_ptr():
            self.obs.copy_(obs)
        if self.graph is not None:
            self.graph.replay()
        else:
            self._forward()
        return self.logits, self.values


class NetworkSearch:
    """AlphaZeroMCTS.search (mcts.py:197-280) for the engine's G games with a NETWORK evaluator, one CUDA graph per
    simulation step: { gmz_select -> folded network -> gmz_expand_backup } -- the reference's per-simulation round trip
    (mcts.py:253 -> workers.py:339-355: pickle, queue, H2D, forward, D2H, queue, unpickle) collapsed into one graph
    launch with nothing leaving the device.  With dtype = bfloat16 the select writes its leaf observations directly as
    bf16 NHWC, the network's input format.  Create the engine with accum_dtype="float32": the network returns float32
    values, and that is the dtype the reference's tree then accumulates in (SURVEY App. A.7)."""

    def __init__(self, engine, net, dtype=torch.bfloat16, graph=True, graph_warmup=2):
        if engine.mode != "AlphaZero":
            raise ValueError("NetworkSearch drives an AlphaZero-mode engine (MuZero mode: muzero.MuZeroDeviceSearch)")
        self.e = engine
        self.obs = engine.obs_buffer_bf16() if dtype == torch.bfloat16 else engine.leaf_obs
        self.ev = DeviceEvaluator(net, self.obs, dtype=dtype, graph=False)
        self.use_graph, self.graph_warmup, self.graph = bool(graph), int(graph_warmup), None
        self._launches_per_step = 0

    def update_weights(self, state_dict):
        self.ev.update_weights(state_dict)           # in place: a captured graph keeps replaying against the same buffers

    def _step(self):
        e = self.e
        e.select(out=self.obs)
        self.ev._forward()
        e.expand_backup(self.ev.logits, self.ev.values)

    def _capture(self):
        e = self.e
        n0 = e.launches
        torch.cuda.synchronize(e.device)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=capture_stream(e.device)):
            self._step()
        self._launches_per_step = e.launches - n0
        e.launches = n0                                # capturing launched nothing

    @torch.no_grad()
    def search(self, gumbel, num_simulations=None):
        """One search for every game from the engine's current roots; follow with engine.finalize()."""
        e = self.e
        e.root_obs(self.obs)
        self.ev._forward()
        e.root_expand(self.ev.logits, self.ev.values, gumbel)
        steps = (e.S if num_simulations is None else int(num_simulations)) - 1
        done = 0
        while done < steps:
            if self.use_graph and self.graph is None and done >= self.graph_warmup:
                self._capture()
            if self.graph is not None:
                self.graph.replay()
                e.launches += self._launches_per_step
            else:
                self._step()
            done += 1
        return done
