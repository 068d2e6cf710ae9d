"""Pick the checker for a model: oracle/_ref (the unmodified reference C, prebuilt or built from its sources,
oracle/ref.py) when available, else the stored outputs of tests/golden/stored.npz (kind 'stored', tests/stored.py)."""
from oracle import ref
from tests.stored import Stored


class _Ref:
    kind = "reference"

    def __init__(self, model):
        self.r = ref.Reference(model)

    def solve(self):
        return self.r.solve()

    def simulate(self, M, D, init, rs, rndtype=0):
        return self.r.simulate(M, D, init, rs, rndtype)

    @property
    def seconds(self):
        return self.r.last_seconds


def ref_available(model) -> bool:
    return ref.build(model) is not None


def oracle_for(model, prefer="reference", whole=False):
    """``whole``: a stored solution keeps every row of every cell (for tests that inspect the rows)."""
    model.prepare()
    if prefer == "reference" and ref_available(model):
        return _Ref(model)
    return Stored(model, whole)
