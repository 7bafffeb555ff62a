"""The designed ReSeg network: backbone -> 2 x ReNet -> dense multi-head attention over the
1/4-resolution map -> two transposed-convolution up-samplings with skips -> semantic logits and
the per-pixel instance embedding.

Reference: /root/reference/code/lib/archs/reseg.py:13-40 documents exactly this model (VGG16 skip
base, two ReNet layers, two transposed convolutions, semantic + instance heads) although the tree
ships a UNet + hard-attention decoder whose instance loss is NaN and whose inference branch raises
(SURVEY.md section 0, R2/R4/R5).  The hot path -- ReNet sweeps, attention, and the embedding map
that feeds DiscriminativeLoss / clustering -- is the B200-native part; the convolutional backbone
and heads are stock cuDNN layers (out of scope, SURVEY.md section 2).

`forward(training, images, ...)` keeps the reference's calling convention (reseg.py:106) and
returns `(sem_seg_logits, ins_seg_embedding)`, which is what `Model.predict` unpacks
(lib/model.py:480-481).

`ReSeg(..., count_head=True)` adds the instance-count branch that reseg.py:13-40 documents as the third head and the
reference tree never builds; the layer list in `CountBranch` is this project's specification (its float64
restatement, the oracle of the tests, is oracle/count_head_ref.py).  `forward` then returns a third element,
`CountFeatures`, whose `evaluate(n_objects)` runs the fused tail (count_head.py).
"""
import torch
import torch.nn as nn

from .attention import MultiHeadAttention
from .count_head import count_tail
from .pointwise import ConvBiasAct, ConvTransposeBiasAct, MaxPool2x2, pixel_heads, thin_linear
from .renet import ReNet


class SkipVGG16(nn.Module):
    """First three VGG16 stages with skips (/root/reference/code/lib/archs/modules/vgg16.py:82-140):
    returns (256 ch @ 1/4, skip 64 ch @ 1/1, skip 128 ch @ 1/2).  Random init (no network access)."""

    def __init__(self, n_input=3):
        super(SkipVGG16, self).__init__()
        self.n_filters = 256

        def block(cin, cout, n):
            layers = []
            for i in range(n):
                # bias + ReLU run as one in-place epilogue kernel (pointwise.py); the Identity keeps the
                # Sequential indices -- and with them the state_dict keys -- of the conv / ReLU pairs
                layers += [ConvBiasAct(cin if i == 0 else cout, cout, 3, padding=1, relu=True), nn.Identity()]
            return nn.Sequential(*layers)

        self.stage1 = block(n_input, 64, 2)
        self.stage2 = block(64, 128, 2)
        self.stage3 = block(128, 256, 3)
        self.pool = MaxPool2x2()

    def forward(self, x):
        # each stage output feeds the next stage through the pool AND a skip connection: pool.with_skip sums the two
        # gradients inside the pooling backward kernel
        p1, s1 = self.pool.with_skip(self.stage1(x))
        p2, s2 = self.pool.with_skip(self.stage2(p1))
        x = self.stage3(p2)
        return x, s1, s2


class EmbeddingPath(nn.Module):
    """The hot path proper: backbone features (N,256,H/4,W/4) -> (N, 2*n_units + d_model, H/4, W/4).
    ReNet x 2 (persistent GRU scan kernels) then multi-head self-attention over the L = H/4*W/4
    positions (tcgen05 kernel), concatenated to the recurrent features."""

    def __init__(self, n_input=256, n_units=100, n_head=2, d_model=24, d_k=12, d_v=12, attn_dropout=0.0, dropout=0.0):
        super(EmbeddingPath, self).__init__()
        self.renet1 = ReNet(n_input, n_units)
        self.renet2 = ReNet(2 * n_units, n_units)
        self.attn_in = nn.Linear(2 * n_units, d_model)
        self.attention = MultiHeadAttention(n_head, d_model, d_k, d_v, dropout=dropout, attn_dropout=attn_dropout)
        self.n_out = 2 * n_units + d_model

    def forward(self, feats, fg_mask=None):
        x = self.renet1(feats)
        x = self.renet2(x)                       # (N, 2n, h, w), channels_last memory
        n, c, h, w = x.shape
        tok = x.permute(0, 2, 3, 1).reshape(n, h * w, c)   # no copy: channels_last
        a = thin_linear(tok, self.attn_in)
        mask = None
        if fg_mask is not None:                  # (N, h, w) 1 = foreground: attend to foreground keys only
            mask = (fg_mask.reshape(n, 1, h * w) == 0)
        a, _ = self.attention(a, a, a, mask=mask)
        out = torch.cat([tok, a], dim=2).reshape(n, h, w, -1).permute(0, 3, 1, 2)
        return out


class CountBranch(nn.Module):
    """`ins_cls_cnn`, the convolutions of the instance-count branch over the EmbeddingPath output y (N, C, H/4, W/4):

        pool1 MaxPool2x2 -> conv1 3x3 C->64 +ReLU -> conv2 3x3 64->64 +ReLU -> pool2 MaxPool2x2
        -> conv3 3x3 64->64 +ReLU -> conv4 3x3 64->64 (bias + ReLU in the fused tail, count_head.py)

    `forward` takes pool1's output (ReSeg pools y with the skip to upsampling1, so that both gradients of y are summed in
    the pooling backward kernel) and returns conv3's output; conv4 is only a parameter holder for the tail."""

    def __init__(self, n_input, n_filters=64):
        super(CountBranch, self).__init__()
        self.pool1 = MaxPool2x2()
        self.conv1 = ConvBiasAct(n_input, n_filters, 3, padding=1, relu=True)
        self.conv2 = ConvBiasAct(n_filters, n_filters, 3, padding=1, relu=True)
        self.pool2 = MaxPool2x2()
        self.conv3 = ConvBiasAct(n_filters, n_filters, 3, padding=1, relu=True)
        self.conv4 = nn.Conv2d(n_filters, n_filters, 3, padding=1)

    def forward(self, x):
        return self.conv3(self.pool2(self.conv2(self.conv1(x))))


class CountRegressor(nn.Module):
    """`ins_cls_out`: global average pool -> linear n_filters -> 1 -> sigmoid (all inside the fused tail)."""

    def __init__(self, n_filters=64):
        super(CountRegressor, self).__init__()
        self.linear = nn.Linear(n_filters, 1)


class CountFeatures(object):
    """conv3's output of the count branch and the layers of its tail.  evaluate(n_objects=None) -> count_head.CountOutput
    (loss, s, n_pred, pooled, y): s in (0, 1) is the predicted count / K, n_pred = clamp(round(s K), 1, K) int32;
    with integer targets n_objects (N,) the loss mean_b (s_b - n_objects_b / K)^2 is computed and differentiable."""

    def __init__(self, x, conv4, linear, max_n_objects):
        self.x, self.conv4, self.linear, self.max_n_objects = x, conv4, linear, max_n_objects

    def evaluate(self, n_objects=None):
        return count_tail(self.x, self.conv4, self.linear, self.max_n_objects, n_objects)


class ReSeg(nn.Module):
    """See module docstring.  Argument names follow reseg.py:52-55."""

    def __init__(self, n_classes, use_instance_seg=True, pretrained=False, use_coordinates=False,
                 use_wae=False, usegpu=True, training=True, n_input=3, n_embedding=24,
                 n_units=100, n_head=2, d_k=12, d_v=12, count_head=False, max_n_objects=None):
        super(ReSeg, self).__init__()
        if pretrained:
            raise ValueError("pretrained VGG16 weights cannot be downloaded here; load a state_dict instead")
        if count_head and not (max_n_objects and 1 <= int(max_n_objects) <= 254):
            raise ValueError("count_head=True needs max_n_objects in 1..254, got %r" % (max_n_objects,))
        self.n_classes = n_classes
        self.use_instance_seg = use_instance_seg
        self.base = SkipVGG16(n_input)
        self.path = EmbeddingPath(self.base.n_filters, n_units, n_head, n_embedding, d_k, d_v)
        c = self.path.n_out
        # transposed convolutions with their ReLU (reseg.py:117-121) fused into the epilogue kernel
        self.upsampling1 = ConvTransposeBiasAct(c, 100, kernel_size=(2, 2), stride=(2, 2), relu=True)
        self.relu1 = nn.Identity()
        self.upsampling2 = ConvTransposeBiasAct(100 + 128, 50, kernel_size=(2, 2), stride=(2, 2), relu=True)
        self.relu2 = nn.Identity()
        self.sem_seg_output = ConvBiasAct(50 + 64, n_classes, kernel_size=(1, 1), stride=(1, 1))
        if use_instance_seg:
            self.ins_seg_output = ConvBiasAct(50 + 64, n_embedding, kernel_size=(1, 1), stride=(1, 1))
        self.count_head = bool(count_head)
        if self.count_head:
            self.max_n_objects = int(max_n_objects)
            self.ins_cls_cnn = CountBranch(c)
            self.ins_cls_out = CountRegressor()

    def forward(self, training, *_input):
        """-> (sem_seg_logits, ins_seg_embedding), plus CountFeatures with the count head."""
        x = _input[0]
        if self.count_head and (x.shape[2] < 16 or x.shape[3] < 16):
            raise ValueError("the count head pools the 1/4-resolution map twice: input height and width must be >= 16, "
                             "got %dx%d" % (x.shape[2], x.shape[3]))
        feats, s1, s2 = self.base(x)
        y = self.path(feats)
        count = None
        if self.count_head:
            p, y = self.ins_cls_cnn.pool1.with_skip(y)
            count = CountFeatures(self.ins_cls_cnn(p), self.ins_cls_cnn.conv4, self.ins_cls_out.linear, self.max_n_objects)
        y = self.relu1(self.upsampling1(y))
        y = torch.cat((y, s2), dim=1)
        y = self.relu2(self.upsampling2(y))
        # both 1x1 heads in one pass over (y | s1) -- the concatenation is never materialised -- straight to the NCHW
        # planes the loss / clustering kernels read
        if self.use_instance_seg:
            out = pixel_heads(y, s1, self.sem_seg_output, self.ins_seg_output)
        else:
            sem_seg_out, _ = pixel_heads(y, s1, self.sem_seg_output)
            out = sem_seg_out, sem_seg_out.argmax(1, keepdim=True).float()
        return out if count is None else (out[0], out[1], count)
