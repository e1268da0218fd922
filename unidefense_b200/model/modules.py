"""Hot-path nn.Modules with the reference's names, constructor arguments and state_dict keys,
computing through the sm_100a kernels (unidefense_b200.ops).

Reference: model/modules.py (Classifier :24-32, FrequencyDynamicFilter :79-105,
SpatialDynamicFilter :108-134, FrequencyStyleTransfer :35-55, SpatialStyleTransfer :58-76,
random_noise :7-12, random_blur :15-16, downscale :19-21) and the decoder Sequentials of
model/unidefense.py:59-102 / :284-308 / :464-500.

The dense projections (layer1 convs, decoder convs) are library calls (cuDNN); everything
between them -- InstanceNorm+activation, BatchNorm statistics/apply, channel mean/max, the 1x1
mask conv, sigmoid, mask*x, tanh -- runs in our fused kernels.  Each module keeps a real
nn.Conv2d / nn.BatchNorm2d / nn.InstanceNorm2d child as the parameter holder so that
SyncBatchNorm.convert_sync_batchnorm, DDP, weight-decay grouping and strict state_dict loading
(engine/forgery_engine.py:142-154,:208) see the same tree as with the reference.
"""

import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F

from .. import ops


class MemoryEfficientSwish(nn.Module):
    """Activation marker of the EfficientNet variant (model/efficientnet/utils.py:80-82).  Inside the
    fused blocks it only selects the swish epilogue; called directly it is x*sigmoid(x)."""

    def forward(self, x):
        return F.silu(x)


def act_name(act_module) -> str:
    if isinstance(act_module, nn.ReLU):
        return "relu"
    if isinstance(act_module, (MemoryEfficientSwish, nn.SiLU)):
        return "swish"
    raise ValueError(f"unsupported activation {type(act_module).__name__} (swish / relu)")


class Classifier(nn.Module):
    """model/modules.py:24-32."""

    def __init__(self, depth=512, num_classes=2):
        super().__init__()
        self.fc = nn.Linear(depth, num_classes)
        self.fc.weight.data.normal_(0, 0.01)
        self.fc.bias.data.fill_(0.0)

    def forward(self, x):
        return self.fc(x)


class DecoderBlock(nn.Sequential):
    """One dec_block{i}: the reference's Sequential layout (conv, InstanceNorm2d, act)* [+ conv, Tanh],
    same child indices, but every (InstanceNorm2d, act) pair runs as ONE single-pass kernel and Tanh
    as our epilogue kernel.  `forward_with_mean` also returns mean_hw(out) -- the triplet feature
    dec_out.mean([-2,-1]) (model/unidefense.py:232-236) -- from the last fused epilogue."""

    def _run(self, x, want_mean):
        mods = list(self)
        i, ymean = 0, None
        last_norm = max((k for k, m in enumerate(mods) if isinstance(m, nn.InstanceNorm2d)), default=-1)
        while i < len(mods):
            m = mods[i]
            if isinstance(m, nn.InstanceNorm2d):
                if m.track_running_stats:
                    raise RuntimeError("DecoderBlock: InstanceNorm2d with running stats is not on the reference path")
                act = act_name(mods[i + 1])
                take = want_mean and i == last_norm and not any(isinstance(t, nn.Tanh) for t in mods)
                # bf16 in -> bf16 out under autocast (the convolutions on either side emit / consume bf16): no casting passes
                xin = x if x.dtype in (torch.float32, torch.bfloat16) else x.float()
                r = ops.in_act(xin, m.weight, m.bias, act, m.eps, want_mean=take)
                x, ymean = r if take else (r, ymean)
                i += 2
            elif isinstance(m, nn.Tanh):
                x = ops.tanh(x.float())
                i += 1
            else:
                x = m(x)
                i += 1
        if want_mean and ymean is None:
            ymean = x.mean(dim=(-2, -1))
        return x, ymean

    def forward(self, x):
        return self._run(x, False)[0]

    def forward_with_mean(self, x):
        return self._run(x, True)


def make_decoder_block(spec, norm, activation, affine, bias):
    """spec: list of ('c'|'t'|'o', c_in, c_out): Conv3x3+IN+act / ConvT3x3 s2+IN+act / Conv3x3+Tanh."""
    layers = []
    for kind, ci, co in spec:
        if kind == "t":
            layers.append(nn.ConvTranspose2d(ci, co, 3, 2, 1, output_padding=1, bias=bias))
        else:
            layers.append(nn.Conv2d(ci, co, kernel_size=3, stride=1, padding=1, bias=bias))
        if kind == "o":
            layers.append(nn.Tanh())
        else:
            layers.append(norm(co, affine=affine))
            layers.append(activation(inplace=True) if activation is nn.ReLU else activation())
    return DecoderBlock(*layers)


# ------------------------------------------------------------------------------------------
# BatchNorm statistics shared by the two dynamic filters (local or cross-rank)
# ------------------------------------------------------------------------------------------
def _sync_group(bn):
    if isinstance(bn, nn.SyncBatchNorm) and dist.is_available() and dist.is_initialized():
        group = bn.process_group if bn.process_group is not None else dist.group.WORLD
        if dist.get_world_size(group) > 1:
            return group
    return None


def merge_bn_stats(means, m2s, counts):
    """Chan et al. parallel combination of per-rank (mean, M2, count) -> global (mean, M2, count).
    means/m2s [R, C], counts [R]."""
    n = counts.sum()
    mean = (means * counts[:, None]).sum(0) / n
    m2 = (m2s + counts[:, None] * (means - mean) ** 2).sum(0)
    return mean, m2, n


def bn_forward_stats(bn, proj, local=None):
    """-> (mean [C], rstd [C], count, stat_reduce); `count` is a python float locally and a 0-dim DEVICE tensor
    under SyncBatchNorm (no host sync, CUDA-graph capturable).  Training: batch statistics (merged over ranks
    when `bn` is a SyncBatchNorm inside an initialised process group, engine/forgery_engine.py:142)
    and the running-stat update of nn.BatchNorm2d (momentum, unbiased variance).  Eval: running stats."""
    use_batch = bn.training or bn.running_mean is None
    if not use_batch:
        return bn.running_mean, torch.rsqrt(bn.running_var + bn.eps), 0, None
    N, C, h, w = proj.shape
    mean, m2 = local if local is not None else ops.bn_local_stats(proj.detach())   # local: from the GEMM epilogue
    count = float(N * h * w)
    group = _sync_group(bn)
    reduce_fn = None
    if group is not None:
        world = dist.get_world_size(group)
        packed = torch.cat([mean, m2, torch.full((1,), count, device=mean.device, dtype=mean.dtype)])   # fill kernel: no H2D copy
        from ..parallel import default_comm
        comm = default_comm()
        if comm is not None and proj.is_cuda and 2 * C + 1 <= comm.max_count:
            gathered = comm.gather(packed)                       # one NVLink peer-memory kernel (csrc/ud_comm.cu)

            def reduce_fn(t):
                return comm.reduce(t.contiguous())
        else:
            parts = [torch.empty_like(packed) for _ in range(world)]
            dist.all_gather(parts, packed, group=group)          # 2C+1 floats per rank (<= 33 KB): latency-bound
            gathered = torch.stack(parts)

            def reduce_fn(t):
                t = t.contiguous()
                dist.all_reduce(t, group=group)
                return t
        mean, m2, count = merge_bn_stats(gathered[:, :C], gathered[:, C:2 * C], gathered[:, 2 * C])
    var = m2 / count
    if bn.training and bn.track_running_stats and bn.running_mean is not None:
        with torch.no_grad():
            bn.num_batches_tracked += 1
            mom = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
            bn.running_mean.mul_(1 - mom).add_(mean, alpha=mom)
            denom = (count - 1.0).clamp(min=1.0) if torch.is_tensor(count) else max(count - 1.0, 1.0)
            bn.running_var.mul_(1 - mom).add_(m2 / denom, alpha=mom)
    return mean, torch.rsqrt(var + bn.eps), (count if torch.is_tensor(count) else int(count)), reduce_fn


class _DynamicFilter(nn.Module):
    def _mask(self, x, diff, want_out):
        conv, bn, act = self.layer1[0], self.layer1[1], self.layer1[2]
        x = x.float()
        use_batch = bn.training or bn.running_mean is None
        local = None
        if ops.proj_supported(x, conv):
            # layer1[0] on the tensor cores (tcgen05 implicit GEMM); its epilogue already holds the batch statistics
            proj, pm, p2 = ops.proj_conv(x, conv.weight, want_stats=use_batch)
            local = (pm, p2) if use_batch else None
        else:
            proj = conv(x).float()
        mean, rstd, count, reduce_fn = bn_forward_stats(bn, proj, local)
        w2 = self.layer2[0].weight.reshape(-1)
        if self.layer2[0].bias is not None:      # bias=True: a constant-one guide channel carries it
            diff = torch.cat([diff, torch.ones_like(diff[:, :1])], dim=1)
            w2 = torch.cat([w2, self.layer2[0].bias.reshape(1)])
        return ops.dyfi_mask(proj, mean, rstd, bn.weight, bn.bias, diff, w2, x, act_name(act), count, want_out,
                             reduce_fn)

    def forward(self, x, diff):
        mask, out = self._mask(x, diff, True)
        return {"mask": mask, "out": out}

    def mask_only(self, x, diff):
        """mask without materialising mask*x (the caller folds the product into its next kernel)."""
        return self._mask(x, diff, False)[0]


class FrequencyDynamicFilter(_DynamicFilter):
    """model/modules.py:79-105: 1x1 conv 2C->2C + norm + act; [mean_c, max_c, diff(6)] -> 1x1 conv -> sigmoid."""

    def __init__(self, depth, activation, norm, affine, bias) -> None:
        super().__init__()
        self.layer1 = nn.Sequential(nn.Conv2d(depth * 2, depth * 2, 1, bias=bias), norm(depth * 2, affine=affine),
                                    activation())
        self.layer2 = nn.Sequential(nn.Conv2d(8, 1, 1, bias=bias), nn.Sigmoid())


class SpatialDynamicFilter(_DynamicFilter):
    """model/modules.py:108-134: 3x3 conv C->C + norm + act; [mean_c, max_c, diff(3)] -> 1x1 conv -> sigmoid."""

    def __init__(self, depth, activation, norm, affine, bias) -> None:
        super().__init__()
        self.layer1 = nn.Sequential(nn.Conv2d(depth, depth, 3, 1, 1, bias=bias), norm(depth, affine=affine),
                                    activation())
        self.layer2 = nn.Sequential(nn.Conv2d(5, 1, 1, bias=bias), nn.Sigmoid())
        # the 3x3 kernel is stored [Cout, ky, kx, Cin] in memory (channels_last): that IS the K-major B operand of the
        # implicit GEMM, so no per-step weight re-layout.  Shape, state_dict key and values are unchanged.
        conv = self.layer1[0]
        conv.weight.data = conv.weight.data.contiguous(memory_format=torch.channels_last)
