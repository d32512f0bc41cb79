"""Batched per-user fold-in (SURVEY.md section 8f-4): the step right after training in the
reference's serving path.  ``python/app_local/models.py:657-703`` (``ALS_Model.__init__``) fits ONE
user's ``k+1`` unknowns against fixed movie factors with ``numpy.linalg.lstsq`` on the rows
``[movie_factors, 1]``; this does it for many users at once on the GPU: it is exactly one user
half-sweep of the exact-solve path (gathered Gram matrix on the fp64 tensor cores + Cholesky,
csrc/als_gram.cu) started from zero factors.

A user needs at least ``k+1`` usable ratings (models.py:669, :694) -- others are returned as
invalid (NaN rows), like the reference's ``_valid = False``.

Two deliberate differences from ``ALS_Model`` (models.py:669-697):

* the reference counts only the ratings whose movie has ALS factors (it filters through
  ``als_movie_ids`` first); here ``item_ids`` already ARE rows of ``item_factors``, so the caller
  does that filtering when it maps raw movie ids -- the validity test is applied to what is
  passed in;
* a rank-deficient system (``k+1`` or more ratings that do not determine every unknown) gets the
  pivot-skipping Cholesky solution -- undetermined unknowns stay at 0, the rest is solved
  consistently -- where ``numpy.linalg.lstsq`` returns the minimum-norm solution.  Both fit the
  given ratings equally well; the factors differ.  Such users are still reported valid.
"""
import numpy

from . import cpp_ls


def fold_in_users(user_ids, item_ids, ratings, num_users, item_factors, num_item_factors):
    """Least-squares user factors for fixed item factors.

    :param user_ids, item_ids, ratings: COO of the (median-subtracted) ratings of the users to
        fit; user ids zero based in ``[0, num_users)``, item ids index ``item_factors``
    :param item_factors: flat ``num_items * num_item_factors`` array (what ``cpp_ls.als`` returns)
    :return: ``user_factors`` ``float64[num_users, num_item_factors+1]`` (last column = bias; NaN
        rows for invalid users) and the boolean ``valid`` mask
    """
    k = num_item_factors
    user_ids = numpy.ascontiguousarray(user_ids, dtype=numpy.int32)
    item_ids = numpy.ascontiguousarray(item_ids, dtype=numpy.int32)
    ratings = numpy.ascontiguousarray(ratings, dtype=numpy.double)
    item_factors = numpy.ascontiguousarray(item_factors, dtype=numpy.double).reshape(-1)
    num_items = len(item_factors) // k
    valid = numpy.bincount(user_ids, minlength=num_users) >= k + 1
    keep = valid[user_ids]
    with cpp_ls.AlsProblem(user_ids[keep], item_ids[keep], ratings[keep], k, num_users,
                           num_items) as prob:
        prob.set_factors(numpy.zeros(num_users * (k + 1)), item_factors)
        prob.half_sweep(True, 0)
        user_factors, _ = prob.get_factors_synced()
    user_factors = user_factors.reshape(num_users, k + 1)
    user_factors[~valid] = numpy.nan
    return user_factors, valid
