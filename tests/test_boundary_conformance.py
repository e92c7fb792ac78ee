"""The drop-in class keeps the reference's call signatures (SURVEY.md 8b).  The reference's signatures of
RampClusterEnvironment.__init__ / reset / step / is_done are stored in tests/golden/reference_cluster_signatures.json
(name, kind and default of every parameter, read off the unmodified reference with inspect.signature)."""
import inspect
import json
import os

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_cluster_signatures.json')


def test_dropin_class_signatures_match_reference():
    from ddls_b200.host.cluster import RampClusterEnvironment as Mine
    reference = json.load(open(GOLDEN))
    for method in ('__init__', 'reset', 'step', 'is_done'):
        ref = reference[method]
        mine = list(inspect.signature(getattr(Mine, method)).parameters.values())
        assert len(mine) >= len(ref), method
        for r, m in zip(ref, mine):                                # same names, order and defaults; extras only at the end
            r_default = r['default'] if r['has_default'] else inspect.Parameter.empty
            assert (r['name'], r_default, r['kind']) == (m.name, m.default, m.kind.name), (method, r, m)
        for extra in mine[len(ref):]:
            assert extra.default is not inspect.Parameter.empty, (method, extra)
