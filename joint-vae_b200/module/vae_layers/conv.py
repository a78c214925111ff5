"""Conv / deconv stacks from the reference's string specs (module/vae_layers/conv.py:20-244,
conv-models.ini:11-30): "[defaults]CxK+P:S++OP-..." with M/A pooling, U upsampling and '!' conv-in-deconv.

The stacks are nn.Sequential of standard torch layer *containers* (so state_dict keys and shapes equal the
reference's: features.0.weight, imager.3.bias, ...); the engine in ..engine executes them.
"""
import re

from torch import nn

from .misc import activation_layers, Reshape

# conv-models.ini of the reference, features / upsampler sections
features_dict = {
    'vgg11': '[x3-Mx2]64-M-128-M-256-256-M-512-512-M-512-512-M-Ax1',
    'vgg11-a': '[x3-Ax2]64-A-128-A-256-256-A-512-512-A-512-512-A-Ax1',
    'vgg13': '[x3-Mx2]64-64-M-128-128-M-256-256-M-512-512-M-512-512-M-Ax1',
    'vgg16': '[x3-Mx2]64-64-M-128-128-M-256-256-256-M-512-512-512-M-512-512-512-M-Ax1',
    'vgg19': '[x3-Mx2]64-64-M-128-128-M-256-256-256-256-M-512-512-512-512-M-512-512-512-512-M-Ax1',
    'vgg19-a': '[x3-Ax2]64-64-A-128-128-A-256-256-256-256-A-512-512-512-512-A-512-512-512-512-A-Ax1',
    'conv32': '[x5+2]32-32:2-64-64:2-200x7+0',
    'conv32-': '[x3+1]32-32-32-32:2-64-64-64-64:2-200x7+0',
    'conv32+': '[x5+2]32-32:2-64-64:2-128-128:2-200x3+0',
}
upsampler_dict = {
    'deconv32': '[x5+2]64x8+0-64-64:2++1-32-32:2++1-32-!3x5+2',
    'deconv32-': '[x3+1]64x8+0-64-64-64-64:2++1-32-32-32-32:2++1-32-!3x5+2',
    'deconv32+': '[x5+2]128x4+0-128-128:2++1-64-64:2++1-32-32:2++1-32-!3x5+2',
    'ivgg': '[!x3+1-U:2]U-!128-U-!64-U-!32-U-!3',
    'ivgg19': '[!x3+1-U:2]U-!512-!512-!512-!512-U-!512-!512-!512-!512-U-!256-!256-!256-!256-U-!128-!128-U-!64-!64-!3',
    'ivgg11': '[!x3+1-U:2]U-!512-!512-U-!512-!512-U-!256-!256-U-!128-U-!64-!3',
}

_FIELDS = (('out_channels', r'^'), ('kernel_size', r'x'), ('padding', r'\+'), ('stride', r':'))


def parse_conv_layer_name(s, ltype='conv', out_channels=32, kernel_size=5, padding='*', stride=None,
                          output_padding=0, activation='relu', output_activation='linear', where='input'):
    """One token of a spec -> dict(ltype=..., out_channels, kernel_size, padding, stride[, output_padding]).
    Same grammar and defaults as conv.py:20-84: padding '*' = k//2 for convs, 0 for pooling; stride None = 1 for
    (de)convs (pooling then uses its kernel size)."""
    fields = list(_FIELDS)
    if where == 'output':
        fields += [('output_padding', r'\+\+'), ('conv_in_deconv', r'\!')]
        ltype = 'deconv'
    head = s[0].lower()
    if head in 'am':
        ltype, s = head + 'pooling', s[1:]
    elif head == 'u':
        ltype, s = 'upsampler', s[1:]
    p = dict(ltype=ltype, out_channels=out_channels, kernel_size=kernel_size, padding=padding, stride=stride)
    if ltype == 'deconv':
        p['output_padding'] = output_padding
    if ltype.endswith('pooling') or ltype == 'upsampler':
        p.pop('out_channels')
        fields = [f for f in fields if f[0] != 'out_channels']
    for key, delim in fields:
        m = re.search(r'{}(?P<v>[0-9|\*]*)'.format(delim), s)
        if m:
            try:
                p[key] = int(m.group('v'))
            except ValueError:
                p[key] = p.get(key)
    if 'conv_in_deconv' in p:
        p['ltype'] = 'conv'
        p['out_channels'] = p.pop('conv_in_deconv')
        p.pop('output_padding')
    if p.get('padding') == '*':
        p['padding'] = p['kernel_size'] // 2 if ltype == 'conv' else 0
    if p['stride'] is None and ltype.endswith('conv'):
        p['stride'] = 1
    return p


def conv_layer_name(layer):
    if isinstance(layer, (nn.Conv2d, nn.ConvTranspose2d)):
        s = '{}x{}'.format(layer.out_channels, layer.kernel_size[0])
        if layer.padding[0] != layer.kernel_size[0] // 2:
            s += '+{}'.format(layer.padding[0])
        if layer.stride[0] != 1:
            s += ':{}'.format(layer.stride[0])
        return s
    if isinstance(layer, (nn.MaxPool2d, nn.AvgPool2d)):
        s = '{}x{}'.format(str(layer)[0], layer.kernel_size)
        if layer.stride != layer.kernel_size:
            s += ':{}'.format(layer.stride)
        return s
    return 'u:{}'.format(layer.scale_factor)


def find_input_shape(layers_name, wanted_output_shape, input_shape=(1, 1)):
    """Smallest (h, w) the upsampler spec maps to wanted_output_shape (conv.py:107-125)."""
    h, w = input_shape
    while True:
        out = build_de_conv_layers((1, h, w), layers_name, where='output').output_shape[1:]
        if tuple(out) == tuple(wanted_output_shape):
            return (h, w)
        if out[0] > wanted_output_shape[0] or out[1] > wanted_output_shape[1]:
            raise ValueError('Did not find an input shape yielding output size ({}, {}) for {}'.format(
                *wanted_output_shape, layers_name))
        h += int(out[0] < wanted_output_shape[0])
        w += int(out[1] < wanted_output_shape[1])


def build_de_conv_layers(input_shape, layers_name, batch_norm=False, where='input', activation='relu',
                         output_activation='linear', output_distribution='gaussian', pretrained_dict=None):
    """conv.py:128-244: features (where='input') or upsampler (where='output') as an nn.Sequential with
    .name, .input_shape, .output_shape, .shapes."""
    if where == 'input' and layers_name.startswith(('resnet', 'densenet')):
        return ResOrDenseNetFeatures(model_name=layers_name, input_shape=input_shape)
    table = features_dict if where == 'input' else upsampler_dict
    name = layers_name if layers_name in table else None
    spec = table.get(layers_name, layers_name)
    if isinstance(input_shape, int):
        input_shape = (input_shape, 1, 1)
    defaults = {}
    if spec[0] == '[':
        end = spec.find(']')
        for tok in spec[1:end].split('-'):
            d = parse_conv_layer_name(tok, where=where)
            defaults[d.pop('ltype')] = d
        spec = spec[end + 1:]
    tokens = spec.split('-')
    c, h, w = input_shape
    layers, names, shapes = [], [], [input_shape]
    last_act = None
    out_c = c
    for i, tok in enumerate(tokens):
        lt = parse_conv_layer_name(tok, where=where)['ltype']
        p = parse_conv_layer_name(tok, **defaults.get(lt, {}), where=where)
        lt = p.pop('ltype')
        if where == 'output' and i == len(tokens) - 1 and output_distribution == 'categorical':
            p['out_channels'] *= 256
        k, pad, st = p.get('kernel_size'), p.get('padding'), p.get('stride')
        if lt == 'conv':
            layer = nn.Conv2d(c, **p)
            c = out_c = p['out_channels']
            h, w = (h + 2 * pad - k) // st + 1, (w + 2 * pad - k) // st + 1
        elif lt == 'deconv':
            layer = nn.ConvTranspose2d(c, **p)
            c = out_c = p['out_channels']
            op = p['output_padding']
            h, w = (h - 1) * st - 2 * pad + k + op, (w - 1) * st - 2 * pad + k + op
        elif lt.endswith('pooling'):
            layer = (nn.MaxPool2d if lt[0] == 'm' else nn.AvgPool2d)(**p)
            out_c = c
            h = (h + 2 * layer.padding - k) // layer.stride + 1
            w = (w + 2 * layer.padding - k) // layer.stride + 1
        elif lt == 'upsampler':
            layer = nn.UpsamplingNearest2d(scale_factor=st)
            h, w = int(h * st), int(w * st)
        else:
            raise ValueError('unknown layer type {} in {}'.format(lt, tok))
        layers.append(layer)
        if lt.endswith('conv'):
            if batch_norm:
                layers.append(nn.BatchNorm2d(c))
            layers.append(activation_layers[activation](**({'inplace': True} if activation == 'relu' else {})))
            last_act = len(layers) - 1
        names.append(conv_layer_name(layer))
        shapes.append((out_c, h, w))
    out_channels = (out_c,)
    if where == 'output':
        layers[last_act] = activation_layers[output_activation]()
        if output_distribution == 'categorical':
            layers.append(Reshape((256, out_c // 256, h, w)))
            out_channels = (256, out_c // 256)
    conv = nn.Sequential(*layers)
    conv.name = name or '-'.join(names)
    conv.output_shape = (*out_channels, h, w)
    conv.input_shape = input_shape
    conv.shapes = shapes
    if pretrained_dict:
        conv.load_state_dict(pretrained_dict)
        for prm in conv.parameters():
            prm.requires_grad_(False)
    return conv


class ResOrDenseNetFeatures(nn.Sequential):
    """torchvision ResNet/DenseNet minus the fc layer as feature extractor (conv.py:247-272).
    `pretrained` defaults to True like the reference; weights must then be in the local torch hub cache."""

    def __init__(self, model_name='resnet152', input_shape=(3, 32, 32), pretrained=True):
        from torchvision import models
        assert input_shape[0] == 3
        try:
            model = getattr(models, model_name)(weights='DEFAULT' if pretrained else None)
        except Exception as e:      # no network / no cached weights: the reference would stop here
            if not pretrained:
                raise
            import logging
            logging.warning('pretrained weights of %s are not available (%s): random initialisation', model_name,
                            type(e).__name__)
            model = getattr(models, model_name)(weights=None)
            pretrained = False
        modules = list(model.children())
        super().__init__(*modules[:-1])
        self.architecture = {'features': model_name}
        self.pretrained = pretrained
        self.name = model_name
        _, w, h = input_shape
        if model_name.startswith('resnet'):
            w, h = 1, 1
        elif model_name.startswith('densenet'):
            w //= 32
            h //= 32
        self.output_shape = (modules[-1].in_features, w, h)
