"""-m "not gpu": which options combine, over every combination of the descriptor flags the rules read, exp_reg,
B_global and the optional arguments of the ten loss entry points and sfm_host_ctx_create, and over every pair of
ViewSynthesisLoss options.

Without a device a call that breaks no rule returns SFM_E_NO_DEVICE, so the code of every combination is that of the
first rule of RULES it breaks (the order decides the code of a call that breaks several).  The rules are those
include/sfmloss.h states per entry point; every refusal must name one of the options involved."""
import ctypes as C
import itertools

import pytest

B, S, H, W, NS = 2, 2, 64, 208, 4
P = 256                                          # placeholder device pointer: aligned, never dereferenced


@pytest.fixture(scope='module')
def lib():
    import torch
    if torch.cuda.is_available():
        pytest.skip('a combination that passes the checks would launch kernels on placeholder pointers')
    import __graft_entry__ as ge
    ge.build()
    from sfm_learner_chainer_b200 import lib as L
    return L


def _rules(L):
    """(breaks(call), code, names the message may give) in order; `call` is a dict of the call's options."""
    I, N, U = L.SFM_E_INVALID_DESC, L.SFM_E_NULL_POINTER, L.SFM_E_UNSUPPORTED
    F = lambda name: getattr(L, 'SFM_FLAG_' + name)
    flag_names = lambda c, names: ['SFM_FLAG_' + n for n in names if c['flags'] & F(n)]
    return [
        (lambda c: c['vm'] and not c['flags'] & F('VALID_MEAN'), I, lambda c: ['SFM_FLAG_VALID_MEAN']),
        (lambda c: c['vm'] and c['peer'], U, lambda c: ['peer']),
        (lambda c: c['vm'] and c['B_global'] not in (0, B), U, lambda c: ['B_global']),
        (lambda c: c['geo'] and not c['flags'] & F('GEOMETRY_CONSISTENCY'), I, lambda c: ['SFM_FLAG_GEOMETRY_CONSISTENCY']),
        (lambda c: c['mr'] and not c['flags'] & F('MIN_REPROJECTION'), I, lambda c: ['SFM_FLAG_MIN_REPROJECTION']),
        (lambda c: (c['geo'] or c['mr']) and c['exp'], U, lambda c: ['exp_reg']),
        (lambda c: c['geo'] and flag_names(c, ['FULL_RES_MULTISCALE', 'BORDER_PADDING', 'MIN_REPROJECTION']), U,
         lambda c: flag_names(c, ['FULL_RES_MULTISCALE', 'BORDER_PADDING', 'MIN_REPROJECTION'])),
        (lambda c: c['terms'] == 'filled' and not c['flags'] & F('SNIPPET_TERMS'), I, lambda c: ['SFM_FLAG_SNIPPET_TERMS']),
        (lambda c: c['ig'] and not c['flags'] & F('IMAGE_GRADS'), I, lambda c: ['SFM_FLAG_IMAGE_GRADS']),
        (lambda c: c['ig'] and flag_names(c, ['EDGE_AWARE_SMOOTH', 'FULL_RES_MULTISCALE']), U,
         lambda c: flag_names(c, ['EDGE_AWARE_SMOOTH', 'FULL_RES_MULTISCALE'])),
        (lambda c: c['ig'] and c['igrads'] != 'filled', N, lambda c: ['igrads']),
        (lambda c: c['ig'] and not c['grads'], N, lambda c: ['grads']),
        (lambda c: c['need_peer'] and not c['peer'], N, lambda c: ['peer']),
        (lambda c: c['pix'] == 'filled' and c['ig'], U, lambda c: ['igrads']),
        (lambda c: c['peer'], U, lambda c: ['peer']),          # the peer here is never connected
        (lambda c: c['flags'] & F('BORDER_PADDING') and (c['exp'] or c['ig'] or c['dbg']), U,
         lambda c: ['SFM_FLAG_BORDER_PADDING']),
        (lambda c: c['flags'] & F('FULL_RES_MULTISCALE') and c['exp'], U, lambda c: ['exp_reg']),
    ]


LOSS_FLAGS = ('IMAGE_GRADS', 'SNIPPET_TERMS', 'MIN_REPROJECTION', 'GEOMETRY_CONSISTENCY', 'VALID_MEAN', 'EDGE_AWARE_SMOOTH',
              'FULL_RES_MULTISCALE', 'BORDER_PADDING')
HOST_FLAGS = ('FULL_RES_MULTISCALE', 'MEAN_NORM_SMOOTH', 'EDGE_MEAN_ABS', 'EDGE_AWARE_SMOOTH', 'BORDER_PADDING',
              'AXISANGLE_POSE', 'GEOMETRY_CONSISTENCY', 'VALID_MEAN')

# entry point -> the optional arguments it takes, each with the forms enumerated (mr and geo are mandatory and given)
ENTRY_POINTS = {
    'sfm_loss_forward': dict(dbg=(False, True)),
    'sfm_loss_backward': dict(gy=(False, True)),
    'sfm_loss_forward_backward': dict(),
    'sfm_loss_forward_backward_peer': dict(peer=(False, True)),
    'sfm_loss_forward_backward_images': dict(igrads=(None, 'empty', 'filled')),
    'sfm_loss_snippets': dict(terms=(None, 'empty', 'filled'), grads=(False, True), igrads=(None, 'empty', 'filled'),
                              peer=(False, True)),
    'sfm_loss_weighted': dict(terms=(None, 'empty', 'filled'), pix=(None, 'empty', 'filled'), grads=(False, True),
                              igrads=(None, 'empty', 'filled'), peer=(False, True)),
    'sfm_loss_min_reprojection': dict(terms=(None, 'empty', 'filled'), grads=(False, True), peer=(False, True)),
    'sfm_loss_geometry': dict(terms=(None, 'empty', 'filled'), grads=(False, True), peer=(False, True)),
    'sfm_loss_geometry_valid_mean': dict(terms=(None, 'empty', 'filled'), vm=(False, True), grads=(False, True),
                                         peer=(False, True)),
}


def _structs(L):
    inp = L.SfmInputs(P, P, P, (P,) * 4, P, (P,) * 4, P, P)
    g = L.SfmGrads((P,) * 4, P, (P,) * 4)
    geo = L.SfmGeometry()
    for s in range(NS):
        geo.src_disps[s] = P
    pix_filled = L.SfmPixelTerms()
    pix_filled.weights[0] = P
    peer = C.create_string_buffer(4096)                      # a zeroed SfmPeer: not connected
    return dict(inp=C.byref(inp), grads=C.byref(g), dbg=C.byref(L.SfmDebug()), gy=C.c_void_p(P),
                peer=C.cast(peer, C.c_void_p),
                igrads={'empty': C.byref(L.SfmImageGrads()), 'filled': C.byref(L.SfmImageGrads(P, None))},
                terms={'empty': C.byref(L.SfmSnippetTerms()), 'filled': C.byref(L.SfmSnippetTerms(P, P))},
                pix={'empty': C.byref(L.SfmPixelTerms()), 'filled': C.byref(pix_filled)},
                mr=C.byref(L.SfmMinReprojection(1, 0)), geo=C.byref(geo),
                vm=C.byref(L.SfmValidMean(1, 1, 0.0, 0)), keep=(inp, g, geo, pix_filled, peer))


def _invoke(so, ep, d, c, st):
    """Calls entry point `ep` with the arguments of combination `c`."""
    pick = lambda k: st[k][c[k]] if c[k] else None
    gr = st['grads'] if c['grads'] else None
    peer = st['peer'] if c['peer'] else None
    los, ws = C.c_void_p(P), C.c_void_p(P)
    if ep == 'sfm_loss_forward':
        return so.sfm_loss_forward(d, st['inp'], los, st['dbg'] if c['dbg'] else None, ws, None)
    if ep == 'sfm_loss_backward':
        return so.sfm_loss_backward(d, st['inp'], st['gy'] if c['gy'] else None, gr, ws, None)
    if ep == 'sfm_loss_forward_backward':
        return so.sfm_loss_forward_backward(d, st['inp'], los, gr, ws, None)
    if ep == 'sfm_loss_forward_backward_peer':
        return so.sfm_loss_forward_backward_peer(d, st['inp'], los, gr, ws, peer, None)
    if ep == 'sfm_loss_forward_backward_images':
        return so.sfm_loss_forward_backward_images(d, st['inp'], los, gr, pick('igrads'), ws, None)
    if ep == 'sfm_loss_snippets':
        return so.sfm_loss_snippets(d, st['inp'], pick('terms'), los, gr, pick('igrads'), ws, peer, None)
    if ep == 'sfm_loss_weighted':
        return so.sfm_loss_weighted(d, st['inp'], pick('terms'), pick('pix'), los, gr, pick('igrads'), ws, peer, None)
    if ep == 'sfm_loss_min_reprojection':
        return so.sfm_loss_min_reprojection(d, st['inp'], pick('terms'), st['mr'], los, gr, ws, peer, None)
    if ep == 'sfm_loss_geometry':
        return so.sfm_loss_geometry(d, st['inp'], pick('terms'), st['geo'], los, gr, ws, peer, None)
    return so.sfm_loss_geometry_valid_mean(d, st['inp'], pick('terms'), st['geo'], st['vm'] if c['vm'] else None, los, gr,
                                           ws, peer, None)


def _flag_sets(L, names):
    bits = [getattr(L, 'SFM_FLAG_' + n) for n in names]
    for on in itertools.product((0, 1), repeat=len(bits)):
        yield sum(b for b, o in zip(bits, on) if o)


def _check(so, rc, code, names, what, bad):
    msg = so.sfm_last_error().decode()
    if rc != code or not any(n in msg for n in names):
        bad.append('%s: rc %d, expected %d naming one of %s; message %r' % (what, rc, code, names, msg))


@pytest.mark.parametrize('ep', sorted(ENTRY_POINTS))
def test_loss_entry_point_matrix(lib, ep):
    so, L = lib.load(), lib
    rules, st = _rules(L), _structs(L)
    opts = ENTRY_POINTS[ep]
    fixed = dict(dbg=False, gy=False, peer=False, igrads=None, terms=None, pix=None, vm=False,
                 grads=ep in ('sfm_loss_backward', 'sfm_loss_forward_backward', 'sfm_loss_forward_backward_peer',
                              'sfm_loss_forward_backward_images'),
                 mr=ep == 'sfm_loss_min_reprojection', geo=ep in ('sfm_loss_geometry', 'sfm_loss_geometry_valid_mean'),
                 need_peer=ep == 'sfm_loss_forward_backward_peer')
    bad, n = [], 0
    for flags in _flag_sets(L, LOSS_FLAGS):
        for exp_reg, B_global in itertools.product((0.0, 0.2), (0, B, 2 * B)):
            d = C.byref(L.SfmDesc(B, S, H, W, NS, B_global, 0.1, exp_reg, 0.15, flags))
            for forms in itertools.product(*opts.values()):
                c = dict(fixed, flags=flags, exp=exp_reg != 0.0, B_global=B_global, **dict(zip(opts, forms)))
                c['ig'] = ep == 'sfm_loss_forward_backward_images' or c['igrads'] is not None
                code, names = L.SFM_E_NO_DEVICE, ['no CPU fallback']
                for breaks, rule_code, rule_names in rules:
                    if breaks(c):
                        code, names = rule_code, rule_names(c)
                        break
                _check(so, _invoke(so, ep, d, c, st), code, names, repr(c), bad)
                n += 1
    assert not bad, '%d of %d combinations differ, e.g.\n%s' % (len(bad), n, '\n'.join(bad[:20]))


def test_host_ctx_matrix(lib):
    so, L = lib.load(), lib
    unsupported = HOST_FLAGS[:3] + HOST_FLAGS[4:]              # every flag the host-buffer path refuses
    bad = []
    for flags in _flag_sets(L, HOST_FLAGS):
        for exp_reg, B_global in itertools.product((0.0, 0.2), (0, B, 2 * B)):
            d = L.SfmDesc(B, S, H, W, NS, B_global, 0.1, exp_reg, 0.15, flags)
            ctx = C.c_void_p()
            refused = ['SFM_FLAG_' + n for n in unsupported if flags & getattr(L, 'SFM_FLAG_' + n)]
            if flags & L.SFM_FLAG_EDGE_MEAN_ABS and not flags & L.SFM_FLAG_EDGE_AWARE_SMOOTH:
                code, names = L.SFM_E_INVALID_DESC, ['SFM_FLAG_EDGE_MEAN_ABS']
            elif refused:
                code, names = L.SFM_E_UNSUPPORTED, refused
            else:
                code, names = L.SFM_E_NO_DEVICE, ['no CPU fallback']
            _check(so, so.sfm_host_ctx_create(C.byref(d), C.byref(ctx)), code, names, 'flags 0x%x' % flags, bad)
    assert not bad, '\n'.join(bad[:20])


def test_operator_option_pairs(lib):
    """Every pair of ViewSynthesisLoss options, each with the options it needs: an excluded pair among them raises
    ValueError naming both options of that pair; any other combination constructs."""
    from sfm_learner_chainer_b200 import ViewSynthesisLoss as V
    value = dict(exp_reg=0.2, B_global=2 * B, invert_sources=(0,))
    names = sorted({n for pair in V.NEEDS + V.EXCLUDES for n in pair})
    needs = dict(V.NEEDS)
    for a, b in itertools.combinations(names, 2):
        on = {a, b}
        on |= {needs[x] for x in on if x in needs}
        kw = {x: value.get(x, True) for x in on}
        excluded = [(x, y) for x, y in V.EXCLUDES if x in on and y in on]
        if excluded:
            with pytest.raises(ValueError) as e:
                V(**kw)
            assert any(x in str(e.value) and y in str(e.value) for x, y in excluded), (kw, str(e.value))
        else:
            V(**kw)
