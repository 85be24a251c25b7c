"""Model zoo of the DFXP path (``models.py:N`` = /root/reference/models.py:N), as nn.Modules over lbt_b200.dfxp.

Inputs are logical NCHW tensors stored channels_last (= the reference's NHWC placeholder,
models.py:10).  ``Model.forward`` returns the logits; ``Model.loss`` is the mean sparse softmax
cross-entropy of models.py:30-32.  The manual reverse chain of models.py:47-51 is PyTorch autograd
over the layers' custom Functions (each of which quantises its incoming gradient itself).
"""
import torch
import torch.nn as nn

from . import dfxp


class Model(nn.Module):
    """models.py:7-54."""

    def __init__(self, bits, dropout=0.5, weight_decay=0.0, stochastic=False, *, grad_bits=None, seed=0):
        super().__init__()
        self.bits, self.dropout, self.weight_decay, self.grad_bits = bits, dropout, weight_decay, grad_bits
        # `stochastic` is accepted and ignored exactly like the reference: every layer hard-codes
        # stochastic=True (dynamic_fixed_point.py:192-206; SURVEY.md F5)
        self.stochastic = stochastic
        self.runtime = dfxp.Runtime(seed)
        self.layers = nn.Sequential(*self.get_layers())

    def get_layers(self):
        return []

    def forward(self, x):
        return dfxp.run_layers(self.layers, x)       # models.py:22-25, with the conv+BN peephole fusion

    @staticmethod
    def loss(logits, labels):
        return dfxp.softmax_cross_entropy(logits, labels)                                      # models.py:30-32

    def info(self):
        return '\n'.join(getattr(l, 'info', lambda: type(l).__name__)() for l in self.layers)

    def ranges(self):
        return self.runtime.ranges()

    def freeze_bn_statistics(self, flag=True):
        """Freeze (flag=True) or unfreeze the statistics of every BatchNorm2d_q: in training mode they then normalise with
        their running averages and stop updating them, while gamma, beta and the rest of the model keep training — the usual
        late phase of quantisation-aware training.  Eval mode is unaffected.  Returns self."""
        for m in self.modules():
            if isinstance(m, dfxp.BatchNorm2d_q):
                m.freeze_statistics(flag)
        return self

    def _kw(self, **extra):
        kw = dict(weight_decay=self.weight_decay, grad_bits=self.grad_bits, runtime=self.runtime)
        kw.update(extra)
        return kw


class CIFAR10_Model(Model):
    """models.py:155-234: 3 x (5x5 conv + bias, ReLU, 3x3/2 max-pool) + dense 400 + dense 10, dropout (keep prob)
    before conv2, conv3, dense1, softmax."""

    def get_layers(self):
        b = self.bits
        pool = lambda: dfxp.MaxPool_q(3, 2, 'SAME')
        drop = lambda: dfxp.Dropout_q(self.dropout, runtime=self.runtime)
        return [
            dfxp.Conv2d_q(b, 3, 64, 5, 1, 'SAME', **self._kw(name='conv1', input_signed=True)),
            dfxp.ReLU_q(), pool(),
            drop(),
            dfxp.Conv2d_q(b, 64, 128, 5, 1, 'SAME', **self._kw(name='conv2', input_signed=False)),
            dfxp.ReLU_q(), pool(),
            drop(),
            dfxp.Conv2d_q(b, 128, 128, 5, 1, 'SAME', **self._kw(name='conv3', input_signed=False)),
            dfxp.ReLU_q(), pool(),
            dfxp.Flatten_q(128 * 4 * 4),
            drop(),
            dfxp.Linear_q(b, 128 * 4 * 4, 400, **self._kw(name='dense1')),
            dfxp.ReLU_q(),
            drop(),
            dfxp.Linear_q(b, 400, 10, **self._kw(name='softmax')),
        ]


class PI_MNIST_Model(Model):
    """models.py:57-88: 784 -> 1024 -> 1024 -> 10 dense network (input [N, 784])."""

    def get_layers(self):
        b = self.bits
        drop = lambda: dfxp.Dropout_q(self.dropout, runtime=self.runtime)
        return [
            dfxp.Linear_q(b, 784, 1024, **self._kw(name='dense1')), dfxp.ReLU_q(), drop(),
            dfxp.Linear_q(b, 1024, 1024, **self._kw(name='dense2')), dfxp.ReLU_q(), drop(),
            dfxp.Linear_q(b, 1024, 10, **self._kw(name='softmax')),
        ]


class MNIST_Model(Model):
    """models.py:91-152: LeNet-5 on [N, 1, 28, 28]."""

    def get_layers(self):
        b = self.bits
        pool = lambda: dfxp.MaxPool_q(2, 2, 'VALID')
        drop = lambda: dfxp.Dropout_q(self.dropout, runtime=self.runtime)
        return [
            dfxp.Conv2d_q(b, 1, 6, 5, 1, 'SAME', **self._kw(name='conv1', input_signed=True)), dfxp.ReLU_q(), pool(),
            dfxp.Conv2d_q(b, 6, 16, 5, 1, 'VALID', **self._kw(name='conv2', input_signed=False)), dfxp.ReLU_q(), pool(),
            dfxp.Conv2d_q(b, 16, 120, 5, 1, 'VALID', **self._kw(name='conv3', input_signed=False)), dfxp.ReLU_q(),
            dfxp.Flatten_q(120), drop(),
            dfxp.Linear_q(b, 120, 84, **self._kw(name='dense1')), dfxp.ReLU_q(), drop(),
            dfxp.Linear_q(b, 84, 10, **self._kw(name='softmax')),
        ]


class CIFAR10_VGG_Model(Model):
    """models.py:237-368."""

    def get_layers(self):
        b = self.bits
        pool = lambda: dfxp.MaxPool_q(3, 2, 'SAME')
        drop = lambda: dfxp.Dropout_q(self.dropout, runtime=self.runtime)
        conv = lambda n, ci, co, signed=False: dfxp.Conv2d_q(b, ci, co, 3, 1, 'SAME', **self._kw(name=n, input_signed=signed))
        return [
            conv('conv1-1', 3, 128, True), dfxp.ReLU_q(), conv('conv1-2', 128, 128), dfxp.ReLU_q(), pool(),
            drop(), conv('conv2-1', 128, 256), dfxp.ReLU_q(), conv('conv2-2', 256, 256), dfxp.ReLU_q(), pool(),
            drop(), conv('conv3-1', 256, 512), dfxp.ReLU_q(), conv('conv3-2', 512, 512), dfxp.ReLU_q(), pool(),
            dfxp.Flatten_q(512 * 4 * 4),
            drop(), dfxp.Linear_q(b, 512 * 4 * 4, 1024, **self._kw(name='dense1')), dfxp.ReLU_q(),
            drop(), dfxp.Linear_q(b, 1024, 1024, **self._kw(name='dense2')), dfxp.ReLU_q(),
            drop(), dfxp.Linear_q(b, 1024, 10, **self._kw(name='softmax')),
        ]


class CIFAR10_Resnet(Model):
    """models.py:371-450."""

    def __init__(self, bits, num_blocks, block=dfxp.ResidualBlock_q, **kw):
        self.num_blocks, self.block = num_blocks, block
        super().__init__(bits, **kw)

    def _build_blocks(self, channels, num_blocks, stride):
        blocks = []
        for i in range(1, 1 + num_blocks):
            blocks.append(self.block(self.bits, self.channels, channels, 1 if i > 1 else stride,
                                     **self._kw(name='block%d-%d' % (channels, i))))
            self.channels = channels * self.block.expansion
        return blocks

    def get_layers(self):
        self.channels = 16
        b = self.bits
        return [
            dfxp.Conv2d_pq(b, 3, 16, 3, 1, 'SAME', bias=False, **self._kw(name='conv1', input_signed=True)),
            dfxp.BatchNorm2d_q(b, 16, relu=True, **self._kw(name='conv1-bn')),      # + ReLU_q (models.py:414)
        ] + self._build_blocks(16, self.num_blocks[0], 1) \
          + self._build_blocks(32, self.num_blocks[1], 2) \
          + self._build_blocks(64, self.num_blocks[2], 2) + [
            dfxp.AvgPool_q(8, 1),
            dfxp.Flatten_q(64),
            dfxp.Linear_q(b, 64, 10, bias=False, **self._kw(name='softmax')),
        ]


def CIFAR10_Resnet20(bits, dropout=0.5, weight_decay=0.0, stochastic=False, **kw):
    """models.py:453-455."""
    return CIFAR10_Resnet(bits, [3, 3, 3], dfxp.ResidualBlock_q, dropout=dropout, weight_decay=weight_decay,
                          stochastic=stochastic, **kw)


def CIFAR10_Resnet32(bits, **kw):
    return CIFAR10_Resnet(bits, [5, 5, 5], dfxp.ResidualBlock_q, **kw)


def CIFAR10_Resnet44(bits, **kw):
    return CIFAR10_Resnet(bits, [7, 7, 7], dfxp.ResidualBlock_q, **kw)


def CIFAR10_Resnet56(bits, **kw):
    return CIFAR10_Resnet(bits, [9, 9, 9], dfxp.ResidualBlock_q, **kw)


class ImageNet_Resnet(Model):
    """ResNet-18/50 composed from the reference's blocks (they are not in models.py — SURVEY.md F8):
    7x7/2 stem + BN + ReLU + 3x3/2 max-pool, four stages, global average pool, dense."""

    def __init__(self, bits, num_blocks, block, image=224, num_classes=1000, **kw):
        self.num_blocks, self.block, self.image, self.num_classes = num_blocks, block, image, num_classes
        super().__init__(bits, **kw)

    _build_blocks = CIFAR10_Resnet._build_blocks

    def get_layers(self):
        self.channels = 64
        b = self.bits
        final = -(-self.image // 32)
        layers = [
            dfxp.Conv2d_q(b, 3, 64, 7, 2, 'SAME', bias=False, **self._kw(name='conv1', input_signed=True)),
            dfxp.BatchNorm2d_q(b, 64, relu=True, **self._kw(name='conv1-bn')),
            dfxp.MaxPool_q(3, 2, 'SAME'),
        ]
        for ch, n, s in zip((64, 128, 256, 512), self.num_blocks, (1, 2, 2, 2)):
            layers += self._build_blocks(ch, n, s)
        layers += [
            dfxp.AvgPool_q(final, 1),
            dfxp.Flatten_q(self.channels),
            dfxp.Linear_q(b, self.channels, self.num_classes, bias=False, **self._kw(name='softmax')),
        ]
        return layers


def Resnet18(bits, **kw):
    return ImageNet_Resnet(bits, [2, 2, 2, 2], dfxp.ResidualBlock_q, **kw)


def Resnet50(bits, **kw):
    return ImageNet_Resnet(bits, [3, 4, 6, 3], dfxp.ResidualBottleneck_q, **kw)
