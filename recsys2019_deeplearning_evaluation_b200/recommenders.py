"""Recommender-level mirrors: the reference's `.fit()` / `._compute_item_score()` / `.recommend()` API on top of the
CUDA core.  Class names, `fit` keyword arguments and fitted attributes (`W_sparse`, `USER_factors`, `ITEM_factors`, ...)
follow the reference so that the evaluator and the hyper-parameter search can drive them unchanged:

    Base/BaseRecommender.py:14-253                       BaseRecommender (init casts, recommend, seen filter)
    Base/BaseSimilarityMatrixRecommender.py:15-116       _compute_item_score = URM[users] . W_sparse
    Base/BaseMatrixFactorizationRecommender.py:15-102    _compute_item_score = U[users] . V^T (+ biases)
    KNN/ItemKNNCFRecommender.py:31-54, KNN/UserKNNCFRecommender.py:32-54
    GraphBased/P3alphaRecommender.py:34-144, GraphBased/RP3betaRecommender.py:31-154
    SLIM_BPR/Cython/SLIM_BPR_Cython.py:67-183
    MatrixFactorization/Cython/MatrixFactorization_Cython.py:33-190
    MatrixFactorization/PureSVDRecommender.py:20-55
    Base/Incremental_Training_Early_Stopping.py:91-261   epoch loop with periodic validation / best-model snapshot

Scores, the seen-item mask and the top-`cutoff` selection run on the device (csrc/score.cu); the dense score block is
only copied to the host when the caller asks for it (`_compute_item_score`, `return_scores=True`).
"""
import ctypes

import numpy as np
import scipy.sparse as sps

from . import _lib
from .similarity import Compute_Similarity, _as_csr_f32


def _dev_csr(M):
    """CSR scipy matrix -> (indptr, indices, data) int32/int32/float32 CUDA tensors."""
    import torch
    M = sps.csr_matrix(M, dtype=np.float32)
    if not M.has_sorted_indices:
        M = M.sorted_indices()
    dev = torch.device("cuda", torch.cuda.current_device())
    return (torch.from_numpy(np.ascontiguousarray(M.indptr, np.int32)).to(dev),
            torch.from_numpy(np.ascontiguousarray(M.indices, np.int32)).to(dev),
            torch.from_numpy(np.ascontiguousarray(M.data, np.float32)).to(dev))


def _stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class BaseRecommender(object):
    RECOMMENDER_NAME = "Recommender_Base_Class"

    def __init__(self, URM_train, verbose=True):
        self.URM_train = sps.csr_matrix(URM_train.copy(), dtype=np.float32)  # BaseRecommender.py:23-24
        self.URM_train.eliminate_zeros()
        self.URM_train.sort_indices()
        self.n_users, self.n_items = self.URM_train.shape
        self.verbose = verbose
        self.items_to_ignore_flag = False
        self.items_to_ignore_ID = np.array([], dtype=np.int64)
        self._cold_user_mask = np.ediff1d(self.URM_train.indptr) == 0
        self._cold_item_mask = np.bincount(self.URM_train.indices, minlength=self.n_items) == 0
        self._lib = _lib.load()
        self._d_urm = None

    def _print(self, string):
        if self.verbose:
            print("{}: {}".format(self.RECOMMENDER_NAME, string))

    def get_URM_train(self):
        return self.URM_train.copy()

    def set_items_to_ignore(self, items_to_ignore):
        self.items_to_ignore_flag = True
        self.items_to_ignore_ID = np.array(items_to_ignore, dtype=np.int64)

    def reset_items_to_ignore(self):
        self.items_to_ignore_flag = False
        self.items_to_ignore_ID = np.array([], dtype=np.int64)

    def _urm_device(self):
        if self._d_urm is None:
            self._d_urm = _dev_csr(self.URM_train)
        return self._d_urm

    # ---- model hand-off in the reference's archive format (Base/BaseRecommender.py:236-253, Base/DataIO.py) ----------
    def _model_dict(self):
        raise NotImplementedError("BaseRecommender: save_model not implemented")

    def save_model(self, folder_path, file_name=None):
        from .dataio import DataIO
        if file_name is None:
            file_name = self.RECOMMENDER_NAME
        self._print("Saving model in file '{}'".format(folder_path + file_name))
        DataIO(folder_path=folder_path).save_data(file_name=file_name, data_dict_to_save=self._model_dict())
        self._print("Saving complete")

    def load_model(self, folder_path, file_name=None):
        from .dataio import DataIO
        if file_name is None:
            file_name = self.RECOMMENDER_NAME
        self._print("Loading model from file '{}'".format(folder_path + file_name))
        data_dict = DataIO(folder_path=folder_path).load_data(file_name=file_name)
        for attrib_name in data_dict.keys():  # BaseRecommender.py:250-251
            self.__setattr__(attrib_name, data_dict[attrib_name])
        self._model_loaded()
        self._print("Loading complete")

    def _model_loaded(self):
        """Device-side copies are keyed by the identity of the host arrays, so they refresh by themselves."""

    def _apply_feature_weighting(self, feature_weighting):
        """KNN/ItemKNNCFRecommender.py:42-50 / KNN/UserKNNCFRecommender.py:43-51: URM_train is REPLACED by the weighted
        matrix (later scoring uses it too), weighting applied to URM.T (items are the documents)."""
        if feature_weighting == "none":
            return
        from .weighting import okapi_BM_25, TF_IDF
        fn = okapi_BM_25 if feature_weighting == "BM25" else TF_IDF
        self.URM_train = sps.csr_matrix(fn(self.URM_train.astype(np.float32).T).T, dtype=np.float32)
        self.URM_train.sort_indices()
        self._d_urm = None

    # ---- device-side pieces shared by every model -----------------------------------------------------------------
    def _scores_device(self, d_users, items_to_compute=None):
        """[B, n_items] float32 CUDA tensor of raw scores; model specific."""
        raise NotImplementedError("BaseRecommender: compute_item_score not assigned for current recommender")

    def _users_tensor(self, user_id_array):
        import torch
        return torch.from_numpy(np.ascontiguousarray(user_id_array, np.int32)).to(torch.device("cuda", torch.cuda.current_device()))

    def _mask_items(self, scores, items_to_compute, d_users=None, seen=False):
        import torch
        keep = None
        if items_to_compute is not None:
            k = np.zeros(self.n_items, np.uint8)
            k[np.asarray(items_to_compute, dtype=np.int64)] = 1
            keep = torch.from_numpy(k).to(scores.device)
        ptr, idx, _ = self._urm_device()
        _lib.check(self._lib.b200_score_mask_device(
            d_users.data_ptr() if (seen and d_users is not None) else None, scores.shape[0],
            ptr.data_ptr() if seen else None, idx.data_ptr() if seen else None,
            keep.data_ptr() if keep is not None else None, self.n_items, scores.data_ptr(), _stream()))
        return scores

    def _compute_item_score(self, user_id_array, items_to_compute=None):
        """(len(user_id_array), n_items) float32 ndarray, -inf on items outside `items_to_compute`."""
        d_users = self._users_tensor(user_id_array)
        scores = self._scores_device(d_users)
        if items_to_compute is not None:
            self._mask_items(scores, items_to_compute)
        return scores.cpu().numpy()

    def _masked_scores_device(self, d_users, remove_seen_flag=True, items_to_compute=None, remove_custom_items_flag=False):
        """BaseRecommender.py:164-196 on the device: score block with seen / not-to-compute / custom items at -inf."""
        import torch
        scores = self._scores_device(d_users)
        if items_to_compute is not None or remove_seen_flag:
            self._mask_items(scores, items_to_compute, d_users, seen=remove_seen_flag)
        if remove_custom_items_flag and len(self.items_to_ignore_ID):
            scores[:, torch.from_numpy(self.items_to_ignore_ID).to(scores.device)] = float("-inf")
        return scores

    def _topn_device(self, scores, cutoff):
        """[B, cutoff] int32 items / float32 scores CUDA tensors, best first, ties by ascending item id (cutoff <= 1024);
        lists end where the score is -inf."""
        import torch
        items = torch.empty((scores.shape[0], cutoff), dtype=torch.int32, device=scores.device)
        vals = torch.empty((scores.shape[0], cutoff), dtype=torch.float32, device=scores.device)
        _lib.check(self._lib.b200_score_topn_device(scores.data_ptr(), scores.shape[0], self.n_items, cutoff, items.data_ptr(),
                                                    vals.data_ptr(), _stream()))
        return items, vals

    def recommend(self, user_id_array, cutoff=None, remove_seen_flag=True, items_to_compute=None, remove_top_pop_flag=False,
                  remove_custom_items_flag=False, return_scores=False):
        """BaseRecommender.py:131-222 on the device: scores -> seen / custom items to -inf -> per-user top-`cutoff`
        (best first, ties by ascending item id) with -inf entries dropped from the lists."""
        single_user = np.isscalar(user_id_array)
        users = np.atleast_1d(user_id_array)
        if cutoff is None:
            cutoff = self.n_items - 1
        cutoff = int(min(cutoff, self.n_items))
        d_users = self._users_tensor(users)
        scores = self._masked_scores_device(d_users, remove_seen_flag, items_to_compute, remove_custom_items_flag)
        if cutoff <= 1024:
            items, vals = self._topn_device(scores, cutoff)
            items_h, vals_h = items.cpu().numpy(), vals.cpu().numpy()
        else:  # full rankings are host work in the reference too; keep the device scores, sort on the host
            sc = scores.cpu().numpy()
            order = np.lexsort((np.broadcast_to(np.arange(self.n_items), sc.shape), -sc), axis=1)[:, :cutoff]
            items_h, vals_h = order.astype(np.int32), np.take_along_axis(sc, order, axis=1)
        ranking_list = [items_h[r][np.isfinite(vals_h[r])].tolist() for r in range(len(users))]
        if single_user:
            ranking_list = ranking_list[0]
        if return_scores:
            return ranking_list, scores.cpu().numpy()
        return ranking_list


class BaseItemSimilarityMatrixRecommender(BaseRecommender):
    """BaseSimilarityMatrixRecommender.py:62-92: scores = URM[users] . W_sparse."""

    def _model_dict(self):
        return {"W_sparse": self.W_sparse}  # BaseSimilarityMatrixRecommender.py:55

    def _w_device(self):
        if getattr(self, "_d_w_src", None) is not self.W_sparse:
            self._d_w = _dev_csr(self.W_sparse)
            self._d_w_src = self.W_sparse
        return self._d_w

    def _scores_device(self, d_users, items_to_compute=None):
        import torch
        a_ptr, a_idx, a_val = self._urm_device()
        b_ptr, b_idx, b_val = self._w_device()
        out = torch.empty((d_users.shape[0], self.n_items), dtype=torch.float32, device=d_users.device)
        _lib.check(self._lib.b200_score_spmm_device(d_users.data_ptr(), d_users.shape[0], a_ptr.data_ptr(), a_idx.data_ptr(),
                                                    a_val.data_ptr(), b_ptr.data_ptr(), b_idx.data_ptr(), b_val.data_ptr(),
                                                    self.n_items, out.data_ptr(), _stream()))
        return out


class BaseUserSimilarityMatrixRecommender(BaseRecommender):
    """BaseSimilarityMatrixRecommender.py:95-116: scores = W_sparse[users] . URM."""

    def _model_dict(self):
        return {"W_sparse": self.W_sparse}  # BaseSimilarityMatrixRecommender.py:55

    def _scores_device(self, d_users, items_to_compute=None):
        import torch
        if getattr(self, "_d_w_src", None) is not self.W_sparse:
            self._d_w = _dev_csr(self.W_sparse)
            self._d_w_src = self.W_sparse
        a_ptr, a_idx, a_val = self._d_w
        b_ptr, b_idx, b_val = self._urm_device()
        out = torch.empty((d_users.shape[0], self.n_items), dtype=torch.float32, device=d_users.device)
        _lib.check(self._lib.b200_score_spmm_device(d_users.data_ptr(), d_users.shape[0], a_ptr.data_ptr(), a_idx.data_ptr(),
                                                    a_val.data_ptr(), b_ptr.data_ptr(), b_idx.data_ptr(), b_val.data_ptr(),
                                                    self.n_items, out.data_ptr(), _stream()))
        return out


class ItemKNNCFRecommender(BaseItemSimilarityMatrixRecommender):
    RECOMMENDER_NAME = "ItemKNNCFRecommender"
    FEATURE_WEIGHTING_VALUES = ["BM25", "TF-IDF", "none"]

    def fit(self, topK=50, shrink=100, similarity="cosine", normalize=True, feature_weighting="none", **similarity_args):
        """KNN/ItemKNNCFRecommender.py:31-54."""
        self.topK, self.shrink = topK, shrink
        if feature_weighting not in self.FEATURE_WEIGHTING_VALUES:
            raise ValueError("Value for 'feature_weighting' not recognized. Acceptable values are {}, provided was '{}'".format(
                self.FEATURE_WEIGHTING_VALUES, feature_weighting))
        self._apply_feature_weighting(feature_weighting)
        sim = Compute_Similarity(self.URM_train, shrink=shrink, topK=topK, normalize=normalize, similarity=similarity,
                                 **similarity_args)
        self.W_sparse = sps.csr_matrix(sim.compute_similarity(), dtype=np.float32)
        sim.compute_similarity_object._dealloc()


class UserKNNCFRecommender(BaseUserSimilarityMatrixRecommender):
    RECOMMENDER_NAME = "UserKNNCFRecommender"
    FEATURE_WEIGHTING_VALUES = ["BM25", "TF-IDF", "none"]

    def fit(self, topK=50, shrink=100, similarity="cosine", normalize=True, feature_weighting="none", **similarity_args):
        """KNN/UserKNNCFRecommender.py:32-54: the same kernel on URM^T (columns = users)."""
        self.topK, self.shrink = topK, shrink
        if feature_weighting not in self.FEATURE_WEIGHTING_VALUES:
            raise ValueError("Value for 'feature_weighting' not recognized. Acceptable values are {}, provided was '{}'".format(
                self.FEATURE_WEIGHTING_VALUES, feature_weighting))
        self._apply_feature_weighting(feature_weighting)
        sim = Compute_Similarity(self.URM_train.T.tocsr(), shrink=shrink, topK=topK, normalize=normalize, similarity=similarity,
                                 **similarity_args)
        self.W_sparse = sps.csr_matrix(sim.compute_similarity(), dtype=np.float32)
        sim.compute_similarity_object._dealloc()


class _GraphFilterMixin(object):
    def _filter_urm_in_place(self, min_rating, implicit):
        """P3alphaRecommender.py:47-51 / RP3betaRecommender.py:44-48 mutate self.URM_train: ratings below `min_rating` are
        dropped (and the rest binarised when `implicit`), so the later scoring (URM[users] . W) and the seen-item
        filter use the filtered matrix too."""
        if min_rating > 0:
            self.URM_train.data[self.URM_train.data < min_rating] = 0
            self.URM_train.eliminate_zeros()
            if implicit:
                self.URM_train.data = np.ones(self.URM_train.data.size, dtype=np.float32)
            self._d_urm = None  # the device copy of the profiles follows the host matrix


class P3alphaRecommender(_GraphFilterMixin, BaseItemSimilarityMatrixRecommender):
    RECOMMENDER_NAME = "P3alphaRecommender"

    def fit(self, topK=100, alpha=1.0, min_rating=0, implicit=False, normalize_similarity=False):
        from .graph import p3_similarity
        self.topK, self.alpha, self.min_rating, self.implicit, self.normalize_similarity = topK, alpha, min_rating, implicit, normalize_similarity
        self._filter_urm_in_place(min_rating, implicit)
        self.W_sparse = p3_similarity(self.URM_train, topK=topK, alpha=alpha, beta=0.0, normalize_similarity=normalize_similarity)


class RP3betaRecommender(_GraphFilterMixin, BaseItemSimilarityMatrixRecommender):
    RECOMMENDER_NAME = "RP3betaRecommender"

    def fit(self, alpha=1.0, beta=0.6, min_rating=0, topK=100, implicit=False, normalize_similarity=True):
        from .graph import p3_similarity
        self.alpha, self.beta, self.min_rating, self.topK, self.implicit, self.normalize_similarity = alpha, beta, min_rating, topK, implicit, normalize_similarity
        self._filter_urm_in_place(min_rating, implicit)
        self.W_sparse = p3_similarity(self.URM_train, topK=topK, alpha=alpha, beta=beta, normalize_similarity=normalize_similarity)


class Incremental_Training_Early_Stopping(object):
    """Base/Incremental_Training_Early_Stopping.py:91-261, same control flow: run epochs, every `validation_every_n`
    epochs prepare the model, evaluate `validation_metric` with `evaluator_object.evaluateRecommender(self)`, keep the
    best snapshot, stop after `lower_validations_allowed` non-improving validations."""

    def _train_with_early_stopping(self, epochs_max, epochs_min=0, validation_every_n=None, stop_on_validation=False,
                                   validation_metric=None, lower_validations_allowed=None, evaluator_object=None,
                                   algorithm_name="Incremental_Training_Early_Stopping"):
        # :147-157, same conditions and messages
        assert epochs_max >= 0, "{}: Number of epochs_max must be >= 0, passed was {}".format(algorithm_name, epochs_max)
        assert epochs_min >= 0, "{}: Number of epochs_min must be >= 0, passed was {}".format(algorithm_name, epochs_min)
        assert epochs_min <= epochs_max, "{}: epochs_min must be <= epochs_max, passed are epochs_min {}, epochs_max {}".format(
            algorithm_name, epochs_min, epochs_max)
        assert evaluator_object is None or \
            (not stop_on_validation and validation_every_n is not None and validation_metric is not None) or \
            (stop_on_validation and validation_every_n is not None and validation_metric is not None and lower_validations_allowed is not None), \
            "{}: Inconsistent parameters passed, please check the supported uses".format(algorithm_name)
        self.best_validation_metric, lower_validation_count = None, 0
        self.epochs_best, epochs_current, convergence = 0, 0, False
        while epochs_current < epochs_max and not convergence:
            self._run_epoch(epochs_current)
            if evaluator_object is None:  # :174-176: no validation, always keep the latest
                self.epochs_best = epochs_current
            elif (epochs_current + 1) % validation_every_n == 0:
                self._prepare_model_for_validation()
                results_run, _ = evaluator_object.evaluateRecommender(self)
                results_run = results_run[list(results_run.keys())[0]]
                current_metric_value = results_run[validation_metric]
                if not np.isfinite(current_metric_value):  # :194-199: a diverged run must not return as if it had converged
                    if hasattr(self, "_clean_temp_folder") and hasattr(self, "temp_file_folder"):
                        self._clean_temp_folder(temp_file_folder=self.temp_file_folder)
                    assert False, "{}: metric value is not a finite number, terminating!".format(self.RECOMMENDER_NAME)
                if self.best_validation_metric is None or self.best_validation_metric < current_metric_value:
                    self.best_validation_metric = current_metric_value
                    self._update_best_model()
                    self.epochs_best = epochs_current + 1
                    lower_validation_count = 0
                else:
                    lower_validation_count += 1
                if stop_on_validation and lower_validation_count >= lower_validations_allowed and epochs_current >= epochs_min:
                    convergence = True
            epochs_current += 1
        if evaluator_object is None:  # :239-242 no validation: the last model is the best model (epochs_best stays epochs_max-1)
            self._prepare_model_for_validation()
            self._update_best_model()


class BaseMatrixFactorizationRecommender(BaseRecommender):
    """BaseMatrixFactorizationRecommender.py:15-102: scores = U[users] . V^T (+ global + user + item bias)."""

    def _model_dict(self):  # BaseMatrixFactorizationRecommender.py:88-96
        d = {"USER_factors": self.USER_factors, "ITEM_factors": self.ITEM_factors, "use_bias": self.use_bias}
        if self.use_bias:
            d["ITEM_bias"], d["USER_bias"], d["GLOBAL_bias"] = self.ITEM_bias, self.USER_bias, self.GLOBAL_bias
        return d

    def __init__(self, URM_train, verbose=True):
        super(BaseMatrixFactorizationRecommender, self).__init__(URM_train, verbose=verbose)
        self.use_bias = False

    def _factors_device(self):
        import torch
        # the source arrays themselves are kept (ids can be recycled after a re-fit)
        src = getattr(self, "_d_f_src", None)
        if src is None or src[0] is not self.USER_factors or src[1] is not self.ITEM_factors:
            dev = torch.device("cuda", torch.cuda.current_device())
            U = torch.from_numpy(np.ascontiguousarray(self.USER_factors, np.float32)).to(dev)
            V = torch.from_numpy(np.ascontiguousarray(self.ITEM_factors, np.float32)).to(dev)
            VT = torch.empty((V.shape[1], V.shape[0]), dtype=torch.float32, device=dev)
            _lib.check(self._lib.b200_transpose_device(V.data_ptr(), V.shape[0], V.shape[1], VT.data_ptr(), _stream()))
            biases = None
            if self.use_bias:
                biases = tuple(torch.from_numpy(np.ascontiguousarray(np.atleast_1d(b), np.float32)).to(dev)
                               for b in (self.USER_bias, self.ITEM_bias, self.GLOBAL_bias))
            self._d_f, self._d_f_src = (U, VT, biases), (self.USER_factors, self.ITEM_factors)
        return self._d_f

    def _scores_device(self, d_users, items_to_compute=None):
        import torch
        U, VT, biases = self._factors_device()
        out = torch.empty((d_users.shape[0], self.n_items), dtype=torch.float32, device=d_users.device)
        bu = bi = mu = None
        if biases is not None:
            bu, bi, mu = (b.data_ptr() for b in biases)
        _lib.check(self._lib.b200_score_mf_device(d_users.data_ptr(), d_users.shape[0], U.data_ptr(), VT.data_ptr(), U.shape[1],
                                                  self.n_items, bu, bi, mu, out.data_ptr(), _stream()))
        return out


class PureSVDRecommender(BaseMatrixFactorizationRecommender):
    """MatrixFactorization/PureSVDRecommender.py:20-55: U, Sigma, VT = randomized_svd(URM_train, num_factors, random_state=
    random_seed) on the device (rsvd.py, csrc/rsvd.cu).  Sigma goes to the item side, as the reference stores it:
    USER_factors = U (n_users, k), ITEM_factors = (diag(Sigma) VT)^T (n_items, k), both float32, k = min(num_factors,
    min(URM shape)).  Scores U . (Sigma VT) do not depend on that split.  random_seed=None draws the start from numpy's global
    stream as the reference does."""
    RECOMMENDER_NAME = "PureSVDRecommender"

    def fit(self, num_factors=100, random_seed=None):
        import torch
        from .rsvd import rsvd_device
        self._print("Computing SVD decomposition...")
        r = rsvd_device(self.URM_train, num_factors, random_state=random_seed, scale_item_side=True)
        self.USER_factors, self.ITEM_factors = r.user.cpu().numpy(), r.item.cpu().numpy()
        # the fitted device factors go to the scorer as they are (its item side is the transpose)
        VT = torch.empty((r.item.shape[1], r.item.shape[0]), dtype=torch.float32, device=r.item.device)
        _lib.check(self._lib.b200_transpose_device(r.item.data_ptr(), r.item.shape[0], r.item.shape[1], VT.data_ptr(), _stream()))
        self._d_f, self._d_f_src = (r.user, VT, None), (self.USER_factors, self.ITEM_factors)
        self._print("... Done!")


class _MatrixFactorization_Cython(BaseMatrixFactorizationRecommender, Incremental_Training_Early_Stopping):
    """MatrixFactorization/Cython/MatrixFactorization_Cython.py:19-141."""
    RECOMMENDER_NAME = "MatrixFactorization_Cython_Recommender"

    def __init__(self, URM_train, verbose=True, algorithm_name="MF_BPR"):
        super(_MatrixFactorization_Cython, self).__init__(URM_train, verbose=verbose)
        self.normalize = False
        self.algorithm_name = algorithm_name

    def fit(self, epochs=300, batch_size=1000, num_factors=10, positive_threshold_BPR=None, learning_rate=0.001, use_bias=True,
            sgd_mode="sgd", negative_interactions_quota=0.0, init_mean=0.0, init_std_dev=0.1, user_reg=0.0, item_reg=0.0,
            bias_reg=0.0, positive_reg=0.0, negative_reg=0.0, random_seed=None, sampler="glibc", hogwild=False,
            **earlystopping_kwargs):
        from .mf_epoch import MatrixFactorization_Cython_Epoch
        self.num_factors, self.use_bias, self.sgd_mode = num_factors, use_bias, sgd_mode
        self.positive_threshold_BPR, self.learning_rate = positive_threshold_BPR, learning_rate
        assert 0.0 <= negative_interactions_quota < 1.0, "{}: negative_interactions_quota must be a float value >=0 and < 1.0, provided was '{}'".format(
            self.RECOMMENDER_NAME, negative_interactions_quota)  # MatrixFactorization_Cython.py:49-50
        self.negative_interactions_quota = negative_interactions_quota
        URM_train_positive = self.URM_train
        if self.algorithm_name == "MF_BPR":  # :63-72
            URM_train_positive = self.URM_train.copy()
            if positive_threshold_BPR is not None:
                URM_train_positive.data = URM_train_positive.data >= positive_threshold_BPR
                URM_train_positive.eliminate_zeros()
                assert URM_train_positive.nnz > 0, "MatrixFactorization_Cython: URM_train_positive is empty, positive threshold is too high"
        self.cythonEpoch = MatrixFactorization_Cython_Epoch(
            URM_train_positive, algorithm_name=self.algorithm_name, n_factors=num_factors, learning_rate=learning_rate,
            sgd_mode=sgd_mode, user_reg=user_reg, item_reg=item_reg, bias_reg=bias_reg, positive_reg=positive_reg,
            negative_reg=negative_reg, batch_size=batch_size, use_bias=use_bias, init_mean=init_mean,
            negative_interactions_quota=negative_interactions_quota, init_std_dev=init_std_dev, verbose=self.verbose,
            random_seed=random_seed, sampler=sampler, hogwild=hogwild)
        self._prepare_model_for_validation()
        self._update_best_model()
        self._train_with_early_stopping(epochs, algorithm_name=self.algorithm_name, **earlystopping_kwargs)
        self.USER_factors, self.ITEM_factors = self.USER_factors_best, self.ITEM_factors_best
        if self.use_bias:
            self.USER_bias, self.ITEM_bias, self.GLOBAL_bias = self.USER_bias_best, self.ITEM_bias_best, self.GLOBAL_bias_best
        self.cythonEpoch._dealloc()

    def _prepare_model_for_validation(self):  # :120-127
        self.USER_factors = self.cythonEpoch.get_USER_factors()
        self.ITEM_factors = self.cythonEpoch.get_ITEM_factors()
        if self.use_bias:
            self.USER_bias = self.cythonEpoch.get_USER_bias()
            self.ITEM_bias = self.cythonEpoch.get_ITEM_bias()
            self.GLOBAL_bias = self.cythonEpoch.get_GLOBAL_bias()

    def _update_best_model(self):  # :129-136
        self.USER_factors_best, self.ITEM_factors_best = self.USER_factors.copy(), self.ITEM_factors.copy()
        if self.use_bias:
            self.USER_bias_best, self.ITEM_bias_best, self.GLOBAL_bias_best = self.USER_bias.copy(), self.ITEM_bias.copy(), np.array(self.GLOBAL_bias)

    def _run_epoch(self, num_epoch):
        self.cythonEpoch.epochIteration_Cython()


class MatrixFactorization_BPR_Cython(_MatrixFactorization_Cython):
    """MatrixFactorization_Cython.py:144-161: forces use_bias=False and negative_interactions_quota=0."""
    RECOMMENDER_NAME = "MatrixFactorization_BPR_Cython_Recommender"

    def __init__(self, *pos_args, **key_args):
        super(MatrixFactorization_BPR_Cython, self).__init__(*pos_args, algorithm_name="MF_BPR", **key_args)

    def fit(self, **key_args):
        key_args["use_bias"] = False
        key_args["negative_interactions_quota"] = 0.0
        super(MatrixFactorization_BPR_Cython, self).fit(**key_args)


class MatrixFactorization_FunkSVD_Cython(_MatrixFactorization_Cython):
    """MatrixFactorization_Cython.py:164-176."""
    RECOMMENDER_NAME = "MatrixFactorization_FunkSVD_Cython_Recommender"

    def __init__(self, *pos_args, **key_args):
        super(MatrixFactorization_FunkSVD_Cython, self).__init__(*pos_args, algorithm_name="FUNK_SVD", **key_args)


class MatrixFactorization_AsySVD_Cython(_MatrixFactorization_Cython):
    """MatrixFactorization_Cython.py:194-275: AsymmetricSVD.  The trainer holds two item-side tables (Y = its USER_factors, X =
    its ITEM_factors); the user factors used for scoring are estimated from the profiles, URM . Y / sqrt(profile length)."""
    RECOMMENDER_NAME = "MatrixFactorization_AsySVD_Cython_Recommender"

    def __init__(self, *pos_args, **key_args):
        super(MatrixFactorization_AsySVD_Cython, self).__init__(*pos_args, algorithm_name="ASY_SVD", **key_args)

    def fit(self, **key_args):
        if "batch_size" in key_args and key_args["batch_size"] > 1:  # :217-220
            print("{}: batch_size not supported for this recommender, setting to default value 1.".format(self.RECOMMENDER_NAME))
        key_args["batch_size"] = 1
        super(MatrixFactorization_AsySVD_Cython, self).fit(**key_args)

    def _prepare_model_for_validation(self):  # :226-242
        self.ITEM_factors_Y = self.cythonEpoch.get_USER_factors()
        self.USER_factors = self._estimate_user_factors(self.ITEM_factors_Y)
        self.ITEM_factors = self.cythonEpoch.get_ITEM_factors()
        if self.use_bias:
            self.USER_bias = self.cythonEpoch.get_USER_bias()
            self.ITEM_bias = self.cythonEpoch.get_ITEM_bias()
            self.GLOBAL_bias = self.cythonEpoch.get_GLOBAL_bias()

    def _update_best_model(self):  # :245-253
        super(MatrixFactorization_AsySVD_Cython, self)._update_best_model()
        self.ITEM_factors_Y_best = self.ITEM_factors_Y.copy()

    def _estimate_user_factors(self, ITEM_factors_Y):  # :256-277: the RATINGS weigh the sum here (training sums unweighted rows)
        profile_length_sqrt = np.sqrt(np.ediff1d(self.URM_train.indptr))
        USER_factors = self.URM_train.dot(ITEM_factors_Y)
        nz = profile_length_sqrt > 0
        USER_factors[nz] /= profile_length_sqrt[nz][:, None]
        return USER_factors


class SLIMElasticNetRecommender(BaseItemSimilarityMatrixRecommender):
    """SLIM_ElasticNet/SLIMElasticNetRecommender.py:20-148.  The reference fits one scikit-learn ElasticNet per item on the URM
    with that item's column zeroed (recomputing X^T X each time); here the Gram matrix is formed once on the device (the dense
    mode of the similarity kernel, as for EASE_R) and csrc/slim_enet.cu runs the Gram-matrix coordinate descent of all items,
    one CTA per item, with sklearn's stopping rule in cyclic coordinate order (the reference's order is random and unseeded:
    its own runs differ from each other by as much as this differs from them, tests/test_oracle_elasticnet.py)."""
    RECOMMENDER_NAME = "SLIMElasticNetRecommender"

    def fit(self, l1_ratio=0.1, alpha=1.0, positive_only=True, topK=100, max_iter=100, tol=1e-4):
        import torch
        assert l1_ratio >= 0 and l1_ratio <= 1, "{}: l1_ratio must be between 0 and 1, provided value was {}".format(
            self.RECOMMENDER_NAME, l1_ratio)  # :43
        self.l1_ratio, self.positive_only, self.topK = l1_ratio, positive_only, topK
        n = self.n_items
        G = EASE_R_Recommender._gram_device(self)  # the same X^T X (it only reads URM_train / n_items)
        X = self.URM_train
        diag = torch.from_numpy(np.asarray(X.multiply(X).sum(axis=0), dtype=np.float32).ravel()).to(G.device)
        coefT = torch.empty((n, n), dtype=torch.float32, device=G.device)
        self._n_iter = torch.empty((n,), dtype=torch.int32, device=G.device)
        _lib.check(self._lib.b200_slim_enet_device(G.data_ptr(), diag.data_ptr(), n, self.n_users, float(l1_ratio), float(alpha),
                                                   int(bool(positive_only)), int(max_iter), float(tol), coefT.data_ptr(),
                                                   self._n_iter.data_ptr(), _stream()))
        del G
        from .slim_bpr_epoch import dense_topk_to_sparse
        # :99-107: per item the min(nnz - 1, topK) largest non-zero coefficients; line j of coefT is the model of item j, i.e.
        # column j of W_sparse (:119-121)
        T = dense_topk_to_sparse(coefT, n, min(int(topK), n), along_columns=False, mode=2)
        self.W_sparse = sps.csr_matrix(T.T, dtype=np.float32)


class SLIM_BPR_Cython(BaseItemSimilarityMatrixRecommender, Incremental_Training_Early_Stopping):
    """SLIM_BPR/Cython/SLIM_BPR_Cython.py:48-183 with S dense on the device.  `train_with_sparse_weights=None` (the reference's
    RAM-based auto selection, :85-103) resolves to the dense mode; True runs the tree mode's semantics (slim_bpr_epoch.py)."""
    RECOMMENDER_NAME = "SLIM_BPR_Recommender"

    def fit(self, epochs=300, positive_threshold_BPR=None, train_with_sparse_weights=None, symmetric=True, random_seed=None,
            lambda_i=0.0, lambda_j=0.0, learning_rate=1e-4, topK=200, sgd_mode="adagrad", gamma=0.995, beta_1=0.9,
            beta_2=0.999, sampler="glibc", hogwild=False, **earlystopping_kwargs):
        from .slim_bpr_epoch import SLIM_BPR_Cython_Epoch, similarityMatrixTopK
        self.symmetric, self.train_with_sparse_weights = symmetric, bool(train_with_sparse_weights)
        URM_train_positive = self.URM_train.copy()
        if positive_threshold_BPR is not None:  # SLIM_BPR_Cython.py:112-116
            URM_train_positive.data = URM_train_positive.data >= positive_threshold_BPR
            URM_train_positive.eliminate_zeros()
            assert URM_train_positive.nnz > 0, "SLIM_BPR_Cython: URM_train_positive is empty, positive threshold is too high"
        if topK is not False and topK < 1:  # :138-140
            raise ValueError("TopK not valid. Acceptable values are either False or a positive integer value. Provided value was '{}'".format(topK))
        self.topK, self._topk_fn = topK, similarityMatrixTopK
        self.cythonEpoch = SLIM_BPR_Cython_Epoch(URM_train_positive, train_with_sparse_weights=self.train_with_sparse_weights,
                                                 final_model_sparse_weights=True,
                                                 topK=topK, learning_rate=learning_rate, li_reg=lambda_i, lj_reg=lambda_j,
                                                 symmetric=symmetric, sgd_mode=sgd_mode, verbose=self.verbose, random_seed=random_seed,
                                                 gamma=gamma, beta_1=beta_1, beta_2=beta_2, sampler=sampler, hogwild=hogwild)
        self.S_incremental = self.cythonEpoch.get_S()
        self.S_best = self.S_incremental.copy()
        self._train_with_early_stopping(epochs, algorithm_name=self.RECOMMENDER_NAME, **earlystopping_kwargs)
        self.get_S_incremental_and_set_W()
        self.cythonEpoch._dealloc()

    def _prepare_model_for_validation(self):
        self.get_S_incremental_and_set_W()

    def _update_best_model(self):
        self.S_best = self.S_incremental.copy()

    def _run_epoch(self, num_epoch):
        self.cythonEpoch.epochIteration_Cython()

    def get_S_incremental_and_set_W(self):  # :174-183: dense training applies a COLUMN top-K on top of get_S
        self.S_incremental = self.cythonEpoch.get_S()
        W = self.S_incremental
        if self.topK is not False and not self.train_with_sparse_weights:  # :178-179: the tree mode keeps get_S's row top-K
            from .graph import sparse_column_topk
            W = sparse_column_topk(sps.csr_matrix(W, dtype=np.float32), self.topK)
        self.W_sparse = sps.csr_matrix(W, dtype=np.float32)


class EASE_R_Recommender(BaseItemSimilarityMatrixRecommender):
    """EASE_R/EASE_R_Recommender.py:36-106.  Gram through the dense mode of the similarity kernel, SPD inverse through
    the blocked-Cholesky kernels of csrc/ease.cu; `topK=None` keeps the dense B on the device for scoring."""
    RECOMMENDER_NAME = "EASE_R_Recommender"

    def fit(self, topK=None, l2_norm=1e3, normalize_matrix=False, verbose=True):
        import torch
        self.verbose = verbose
        if normalize_matrix:  # :47-51, sklearn.normalize l2 on rows then columns
            X = self.URM_train.astype(np.float64)
            rn = np.sqrt(np.asarray(X.multiply(X).sum(axis=1)).ravel()); rn[rn == 0] = 1
            X = sps.diags(1.0 / rn).dot(X)
            cn = np.sqrt(np.asarray(X.multiply(X).sum(axis=0)).ravel()); cn[cn == 0] = 1
            self.URM_train = sps.csr_matrix(X.dot(sps.diags(1.0 / cn)), dtype=np.float32)
            self._d_urm = None
        n = self.n_items
        G = self._gram_device()
        _, d_idx, _ = self._urm_device()
        B = torch.empty((n, n), dtype=torch.float32, device=G.device)
        _lib.check(self._lib.b200_ease_from_gram_device(G.data_ptr(), n, d_idx.data_ptr(), self.URM_train.nnz, float(l2_norm), None,
                                                        B.data_ptr(), _stream()))
        del G
        if topK is None:  # :75-78: dense W, scores = URM[users] . W
            self._d_B = B
            self.W_sparse = B.cpu().numpy()
        else:  # :80-82
            from .slim_bpr_epoch import dense_topk_to_sparse
            self._d_B = None
            self.W_sparse = sps.csr_matrix(dense_topk_to_sparse(B, n, topK, along_columns=True, mode=0), dtype=np.float32)

    def _gram_device(self, rows=None):
        """X^T X (EASE_R_Recommender.py:55-56) as a dense [n_items, n_items] fp32 CUDA tensor, from all users or from the
        user rows [rows[0], rows[1]) only (the partial Gram of one rank, dist.make_sharded_ease)."""
        from .similarity import Compute_Similarity_Cython
        n = self.n_items
        X = self.URM_train if rows is None else self.URM_train[rows[0]:rows[1]]
        sim = Compute_Similarity_Cython(X, shrink=0, topK=n if n > 2048 else 0, normalize=False, similarity="cosine")
        G = sim.compute_dense_device(0, n)  # symmetric: orientation is irrelevant
        sim._dealloc()
        return G

    def _model_loaded(self):
        import torch
        self._d_B = None
        if isinstance(self.W_sparse, np.ndarray):  # dense model (topK=None): scoring reads it from the device
            self._d_B = torch.from_numpy(np.ascontiguousarray(self.W_sparse, np.float32)).to(torch.device("cuda", torch.cuda.current_device()))

    def _scores_device(self, d_users, items_to_compute=None):
        if getattr(self, "_d_B", None) is None:
            return super(EASE_R_Recommender, self)._scores_device(d_users, items_to_compute)
        import torch
        n = self.n_items  # dense W (EASE_R_Recommender.py:87-106): out[b, :] = sum over the user's (i, r) of r * B[i, :]
        a_ptr, a_idx, a_val = self._urm_device()
        out = torch.empty((d_users.shape[0], n), dtype=torch.float32, device=d_users.device)
        _lib.check(self._lib.b200_score_spmm_device(d_users.data_ptr(), d_users.shape[0], a_ptr.data_ptr(), a_idx.data_ptr(),
                                                    a_val.data_ptr(), None, None, self._d_B.data_ptr(), n,
                                                    out.data_ptr(), _stream()))
        return out


class IALSRecommender(BaseMatrixFactorizationRecommender, Incremental_Training_Early_Stopping):
    """MatrixFactorization/IALSRecommender.py:19-213.  Factors live on the device in fp64; one `_run_epoch` is two calls
    of the per-row normal-equation kernel (csrc/ials.cu).  Initial factors come from numpy's global RNG exactly like
    :204-210 (seed it before fit() to reproduce a reference run); cold rows keep whatever np.empty gave the reference --
    here zeros."""
    RECOMMENDER_NAME = "IALSRecommender"
    AVAILABLE_CONFIDENCE_SCALING = ["linear", "log"]

    def fit(self, epochs=300, num_factors=20, confidence_scaling="linear", alpha=1.0, epsilon=1.0, reg=1e-3, init_mean=0.0,
            init_std=0.1, **earlystopping_kwargs):
        import torch
        if confidence_scaling not in self.AVAILABLE_CONFIDENCE_SCALING:  # :63-64
            raise ValueError("Value for 'confidence_scaling' not recognized. Acceptable values are {}, provided was '{}'".format(
                self.AVAILABLE_CONFIDENCE_SCALING, confidence_scaling))
        self.num_factors, self.alpha, self.epsilon, self.reg = num_factors, alpha, epsilon, reg
        dev = torch.device("cuda", torch.cuda.current_device())
        self.ITEM_factors = self.num_factors ** -0.5 * np.random.random_sample((self.n_items, self.num_factors))  # :71-72, :204-207
        self.USER_factors = np.zeros((self.n_users, self.num_factors))
        C = self.URM_train.copy()  # :99-123
        if confidence_scaling == "linear":
            C.data = (1.0 + alpha * C.data).astype(np.float32)
        else:
            C.data = (1.0 + alpha * np.log(1.0 + C.data / epsilon)).astype(np.float32)
        C_csc = sps.csc_matrix(C, dtype=np.float32)
        self._d_C = _dev_csr(C)
        self._d_Ct = (torch.from_numpy(np.ascontiguousarray(C_csc.indptr, np.int32)).to(dev),
                      torch.from_numpy(np.ascontiguousarray(C_csc.indices, np.int32)).to(dev),
                      torch.from_numpy(np.ascontiguousarray(C_csc.data, np.float32)).to(dev))
        self._d_warm_users = torch.from_numpy(np.flatnonzero(np.diff(C.indptr) > 0).astype(np.int32)).to(dev)  # :78-82
        self._d_warm_items = torch.from_numpy(np.flatnonzero(np.diff(C_csc.indptr) > 0).astype(np.int32)).to(dev)
        self._d_U = torch.from_numpy(self.USER_factors).to(dev)
        self._d_V = torch.from_numpy(np.ascontiguousarray(self.ITEM_factors)).to(dev)
        self._d_work = torch.empty((num_factors, num_factors), dtype=torch.float64, device=dev)
        self._update_best_model()
        self._train_with_early_stopping(epochs, algorithm_name=self.RECOMMENDER_NAME, **earlystopping_kwargs)
        self.USER_factors, self.ITEM_factors = self.USER_factors_best, self.ITEM_factors_best

    def _half(self, rows, csr, Y, X):
        ptr, idx, conf = csr
        _lib.check(self._lib.b200_ials_half_epoch_device(rows.data_ptr(), rows.shape[0], ptr.data_ptr(), idx.data_ptr(), conf.data_ptr(),
                                                         Y.data_ptr(), Y.shape[0], self.num_factors, float(self.reg), X.data_ptr(),
                                                         self._d_work.data_ptr(), _stream()))

    def _run_epoch(self, num_epoch):  # :137-166
        self._half(self._d_warm_users, self._d_C, self._d_V, self._d_U)
        self._half(self._d_warm_items, self._d_Ct, self._d_U, self._d_V)

    def _prepare_model_for_validation(self):
        self.USER_factors = self._d_U.cpu().numpy()
        self.ITEM_factors = self._d_V.cpu().numpy()

    def _update_best_model(self):
        self._prepare_model_for_validation()
        self.USER_factors_best, self.ITEM_factors_best = self.USER_factors.copy(), self.ITEM_factors.copy()
