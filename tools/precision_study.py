"""CPU study: where does fp16 storage hurt?  Monkeypatches the oracle network so that selected
activations / weights are rounded to fp16 like the native engine does, and replays the golden clip."""
import os, sys
import numpy as np, torch
import torch.nn.functional as F
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tracking-anything-with-deva_b200'))
from oracle import fixtures
from oracle import network as net
from oracle import memory_math as mm
from oracle.core import CoreOracle
from deva.model.param_spec import synthetic_state_dict
torch.set_grad_enabled(False)

FLAGS = dict(enc=True, key=True, maskenc=True, dec=True, up168=True, up84=True, pred=True, gru=True, weights=True)

def rh(x, on=True):
    return x.half().float() if on else x

orig_conv, orig_bn = net._conv, net._bn

def region(name):
    if name.startswith('pixel_encoder'): return 'enc'
    if name.startswith('key_proj'): return 'key'
    if name.startswith('mask_encoder'): return 'gru' if 'sensory_update' in name else 'maskenc'
    if 'sensory_update' in name: return 'gru'
    if name.endswith('.pred'): return 'pred'
    if 'up_8_4' in name: return 'up84'
    if 'up_16_8' in name: return 'up168'
    return 'dec'

def conv(sd, name, x, stride=1, pad=0):
    on = FLAGS[region(name)]
    w = sd[name + '.weight']
    if FLAGS['weights'] and on: w = rh(w)
    y = F.conv2d(rh(x, on), w, sd.get(name + '.bias'), stride=stride, padding=pad)
    # convs followed by BN are rounded after BN; others here
    if name.endswith('pred') or name.startswith('key_proj'): return y
    has_bn = any(k.startswith(name.rsplit('.', 1)[0] + '.bn') for k in ()) 
    return y
def bn(sd, name, x):
    return orig_bn(sd, name, x)
net._conv = conv
net._bn = bn

# persistent state kept in fp16 by the native engine: the per-object sensory (hidden) state, the bank's values,
# and the memory readout handed to the decoder
STATE = dict(sensory=False, values=False, readout=False)
orig_gru, orig_encode_mask, orig_readout = net._gru, net.encode_mask, mm.readout
def gru(values, h, dim):
    return rh(orig_gru(values, rh(h, STATE['sensory']), dim), STATE['sensory'])
def encode_mask(*a, **k):
    v, s = orig_encode_mask(*a, **k)
    return rh(v, STATE['values']), s
def readout(aff, mv):
    return rh(orig_readout(rh(aff, STATE['readout']), rh(mv, STATE['values'])), STATE['readout'])
net._gru = gru
net.encode_mask = encode_mask
mm.readout = readout

def run(tag):
    arrays, meta = fixtures.vos_steps()
    g = {k: torch.from_numpy(v) for k, v in arrays.items()}
    np.random.seed(42)
    core = CoreOracle(synthetic_state_dict(seed=1), meta['config'])
    worst = 0
    T = g['frames'].shape[0]
    for t in range(T):
        if t == 0: p = core.step(g['frames'][t], g['mask0'], [1, 2])
        elif t == 6: p = core.step(g['frames'][t], g['mask6'], [7])
        else: p = core.step(g['frames'][t], end=(t == T - 1))
        worst = max(worst, float((p - g[f'prob_{t:02d}']).abs().max()))
    print(f'{tag:40s} max err {worst:.2e}', flush=True)

if __name__ == '__main__':
    base = dict(FLAGS)
    def only(*names):
        for k in base: FLAGS[k] = False
        for n in names: FLAGS[n] = True
        FLAGS['weights'] = True
    if len(sys.argv) > 1 and sys.argv[1] == 'state':
        nat = ('maskenc', 'dec', 'up168', 'up84', 'gru')  # the native engine: key path + pred precise, rest fp16
        only(*nat); run('native emulation, states fp32')
        for combo in (('sensory',), ('values',), ('readout',), ('sensory', 'values', 'readout')):
            for k in STATE: STATE[k] = k in combo
            only(*nat); run('  + fp16 ' + '+'.join(combo))
        for k in STATE: STATE[k] = False
        only('maskenc', 'dec', 'up168', 'gru'); run('up_8_4 precise')
        only('maskenc', 'dec', 'up84', 'gru'); run('up_16_8 precise')
        only('maskenc', 'up168', 'up84', 'gru'); run('fuser/skip/compress precise')
        only('dec', 'up168', 'up84', 'gru'); run('mask encoder precise')
        only('maskenc', 'dec', 'up168', 'up84'); run('sensory update convs precise')
        sys.exit(0)
    only('maskenc', 'dec', 'up168', 'up84', 'pred', 'gru'); run('key path (enc+key) precise, rest fp16')
    only('maskenc', 'dec', 'up168', 'up84', 'gru'); run('  + pred precise')
    only('maskenc', 'dec', 'up168', 'gru'); run('  + pred, up_8_4 precise')
    only('maskenc', 'gru'); run('  + whole decoder precise')
    only('dec'); run('fp16 only in decoder fuser/skip/compress')
    only('up168'); run('fp16 only in up_16_8')
    only('up84'); run('fp16 only in up_8_4')
    only('pred'); run('fp16 only in pred')
