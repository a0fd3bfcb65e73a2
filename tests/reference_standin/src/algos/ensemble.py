from src.algos.util import Unpatched


class DeepEnsemble(Unpatched):
    pass
