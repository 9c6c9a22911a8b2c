"""recmodel_b200: a B200-native (sm_100a) implementation of the WMF train + top-N path of
titoeb/RecModel behind the reference's own ``WMF`` class API. See DESIGN.md."""
from .wmf_model import WMF, WMFModel  # noqa: F401
from .ease_model import Ease  # noqa: F401
from .knn_model import ItemKNN, UserKNN  # noqa: F401
from .slim_model import SLIM  # noqa: F401
from .rp3beta_model import RP3beta  # noqa: F401
from .utils import split_users, test_coverage, train_test_split_sparse_mat  # noqa: F401

__all__ = ["WMF", "WMFModel", "Ease", "ItemKNN", "UserKNN", "SLIM", "RP3beta", "train_test_split_sparse_mat", "test_coverage",
           "split_users"]
