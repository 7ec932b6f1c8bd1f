"""Drop-in for the p-value arithmetic of DIGDriver/sequence_model/nb_model.py.  The SciPy calls
(scipy.special.betainc, scipy.stats.nbinom.pmf) are replaced by the FP64 kernel K7."""
import numpy as np
import torch

from .. import kernels


def _dev():
    return torch.device("cuda", torch.cuda.current_device())


def normal_params_to_gamma(mu, sigma):
    """Reference :237-241."""
    alpha = mu ** 2 / sigma ** 2
    theta = sigma ** 2 / mu
    return alpha, theta


def _like(ref, values):
    """Return ``values`` as the same kind of object the reference would (Series in -> Series out)."""
    try:
        import pandas as pd
        if isinstance(ref, pd.Series):
            return pd.Series(values, index=ref.index)
    except Exception:
        pass
    if np.ndim(ref) == 0:
        return float(values[0])
    return values


def nb_pvalue_greater_midp(k, alpha, p):
    """UPPER TAIL p-value of a negative binomial with a mid-p correction (reference :271-278):
    0.5 * nbinom.pmf(k, alpha, p) + betainc(k + 1, alpha, 1 - p), evaluated by the GPU kernel."""
    kb, ab, pb = np.broadcast_arrays(np.asarray(k, dtype=np.float64), np.asarray(alpha, dtype=np.float64),
                                     np.asarray(p, dtype=np.float64))
    shape = kb.shape
    out = kernels.nb_pvalue_greater_midp(np.ascontiguousarray(kb).reshape(-1), np.ascontiguousarray(ab).reshape(-1),
                                         np.ascontiguousarray(pb).reshape(-1), _dev()).cpu().numpy()
    for ref in (k, alpha, p):
        if hasattr(ref, "index"):
            return _like(ref, out)
    return out.reshape(shape) if shape else float(out[0])


def get_q_vals(pvals_lst):
    """Benjamini-Hochberg FDR (statsmodels fdrcorrection, method='indep') of reference :340-342."""
    p = np.asarray(pvals_lst, dtype=np.float64)
    n = len(p)
    order = np.argsort(p)
    ranked = p[order] * n / np.arange(1, n + 1)
    q = np.minimum.accumulate(ranked[::-1])[::-1]
    q = np.minimum(q, 1.0)
    out = np.empty(n)
    out[order] = q
    return out


def _variant(mode, k, alpha, p, mu=None):
    """Broadcast (k, alpha, p[, mu]), run dig_nb_pvalue_variant, and hand back what the reference would (a float for
    scalars, a Series for Series arguments, an array otherwise)."""
    args = [np.asarray(x, dtype=np.float64) for x in (k, alpha, p)]
    if mu is not None:
        args.append(np.asarray(mu, dtype=np.float64))
    bc = np.broadcast_arrays(*args)
    shape = bc[0].shape
    flat = [np.ascontiguousarray(b).reshape(-1) for b in bc]
    out = kernels.nb_pvalue_variant(mode, flat[0], flat[1], flat[2], flat[3] if mu is not None else None,
                                    _dev()).cpu().numpy()
    for ref in (k, alpha, p):
        if hasattr(ref, "index") and not callable(ref.index):
            return _like(ref, out)
    return out.reshape(shape) if shape else float(out[0])


def nb_pvalue_greater(k, alpha, p):
    """UPPER TAIL p-value (reference :243-256): 1 for k == 0, else betainc(k, alpha, 1-p) with the pmf as the
    fallback when that underflows to 0."""
    return _variant("greater", k, alpha, p)


def nb_pvalue_greater_midp_DEPRECATED(k, alpha, p):
    """Reference :258-269; for k == 0 its `1 - 0.5 pmf` equals the mid-p expression, so this is nb_pvalue_greater_midp."""
    return _variant("greater_midp", k, alpha, p)


def nb_pvalue_less(k, alpha, p):
    """LOWER TAIL p-value betainc(alpha, k+1, p) (reference :280-283).  The reference computes this value and falls
    off the end of the function (returns None); the value is returned here (SURVEY.md section 8 quirks: not emulated)."""
    return _variant("less", k, alpha, p)


def nb_pvalue_less_midp(k, alpha, p):
    """LOWER TAIL p-value with a mid-p correction (reference :285-296)."""
    return _variant("less_midp", k, alpha, p)


def nb_pvalue_exact(k, alpha, p, mu=None):
    """UPPER or LOWER TAIL p-value of a negative binomial, chosen by whether k is below the expectation
    (reference :298-314).  ``mu`` overrides the expectation alpha (1-p)/p when truthy, as in the reference."""
    if mu is None or (np.ndim(mu) == 0 and not mu):
        kb, ab, pb = np.broadcast_arrays(np.asarray(k, dtype=np.float64), np.asarray(alpha, dtype=np.float64),
                                         np.asarray(p, dtype=np.float64))
        shape = kb.shape
        out = kernels.nb_pvalue_exact(np.ascontiguousarray(kb).reshape(-1), np.ascontiguousarray(ab).reshape(-1),
                                      np.ascontiguousarray(pb).reshape(-1), _dev()).cpu().numpy()
        return out.reshape(shape) if shape else float(out[0])
    return _variant("exact", k, alpha, p, mu)


def nb_pvalue_midp(k, alpha, p, mu=None):
    """Two-sided-by-side mid-p p-value (reference :316-337): lower tail when k < mu, else upper tail."""
    if mu is None:
        return _variant("midp", k, alpha, p)
    return _variant("midp", k, alpha, p, mu)


def tabix_to_dataframe(tbx, chrom, start, end):
    """Rows of a tabix-indexed mutation file in [start, end) as a DataFrame (reference :13-34)."""
    import pandas as pd
    res = [row.split("\t") for row in tbx.fetch(chrom, start, end)]
    if not res or len(res[0]) == 6:
        cols = ['CHROM', 'START', 'END', 'REF', 'ALT', 'ID']
    elif len(res[0]) == 7:
        cols = ['CHROM', 'START', 'END', 'REF', 'ALT', 'ID', 'ANNOT']
    elif len(res[0]) == 8:
        cols = ['CHROM', 'START', 'END', 'REF', 'ALT', 'ID', 'MUT', 'CONTEXT']
    else:
        cols = ['CHROM', 'START', 'END', 'REF', 'ALT', 'ID', 'ANNOT', 'MUT', 'CONTEXT']
    df = pd.DataFrame(res, columns=cols)
    return df.astype(dict(START=int, END=int))


def mutation_freq_conditional(S_mut, S_gen, N):
    """Pr(b | context) = #{b | context} / (N * #{context}) for a Series indexed by (mutation, context) tuples
    (reference :36-55)."""
    ctx = [tup[1] for tup in S_mut.index]
    out = S_mut.astype(float)
    out[:] = S_mut.values / (N * S_gen[ctx].values)
    return out


def mutation_freq_joint(S_mut, S_gen, N):
    """The reference's body is identical to mutation_freq_conditional (:57-77)."""
    return mutation_freq_conditional(S_mut, S_gen, N)


def train_sequence_model(train_idx, f_model, N, key_prefix=None):
    """Context model from the pre-tabulated `mutation_counts` / `genome_counts` tables of f_model restricted to the
    training windows (reference :79-107): (Series of Pr(b | context), {context: sum over b})."""
    from .. import storage
    rows = ['chr{}:{}-{}'.format(r[0], r[1], r[2]) for r in train_idx]
    key_mut = 'mutation_counts' if not key_prefix else key_prefix + "_mutation_counts"
    st = storage.Store(f_model, "r")
    df_mut, df_gen = st.read_table(key_mut), st.read_table('genome_counts')
    S_mut_train = df_mut.loc[rows, :].sum(axis=0)
    S_gen_train = df_gen.loc[rows, :].sum(axis=0)
    Pr = mutation_freq_conditional(S_mut_train, S_gen_train, N)
    d = {}
    for tup, v in zip(Pr.index, Pr.values):          # same left-to-right order as the reference's sum([...])
        d[tup[1]] = d.get(tup[1], 0) + v
    return Pr, d


def expected_mutations_by_context(train_idx, test_idx, f_model, N=1, key_prefix=None):
    """Expected mutations per window from sequence context alone (reference :109-124)."""
    import pandas as pd
    from .. import storage
    _, d_mut = train_sequence_model(train_idx, f_model, N, key_prefix=key_prefix)
    s_mut = pd.Series(d_mut)
    df_gen = storage.Store(f_model, "r").read_table('genome_counts')
    df_exp = (df_gen * s_mut).sum(axis=1)
    tr = ['chr{}:{}-{}'.format(r[0], r[1], r[2]) for r in train_idx]
    te = ['chr{}:{}-{}'.format(r[0], r[1], r[2]) for r in test_idx]
    return df_exp.loc[tr], df_exp.loc[te]


def _mutation_starts(tabix):
    """The reference reads mutations through pysam.TabixFile (absent here): accept a DataFrame with CHROM / START
    columns, a (chrom, start) array pair, or a path to a mutation file readable by data_tools.read_mutation_file.
    Chromosome names come back without a leading 'chr' in every form."""
    import pandas as pd
    if isinstance(tabix, (str, bytes)):
        from ..data_tools import mutation_tools
        tabix = mutation_tools.read_mutation_file(tabix, drop_sex=False)
    if isinstance(tabix, pd.DataFrame):
        chrom, start = tabix.CHROM.values, tabix.START.values
    else:
        chrom, start = tabix
    return (pd.Series(np.asarray(chrom)).astype(str).str.replace("^chr", "", regex=True).values,
            np.asarray(start, dtype=np.int64))


def nb_model(d_pr, idx, mu_lst, sigma_lst, f_tabix, f_fasta, n_up=2, n_down=2, binsize=50, collapse=False):
    """Per-position (binsize=1) or per-bin NB hotspot test over the regions ``idx`` = rows of (CHROM, START, END)
    (reference :188-235): one K8 launch for all regions instead of a Python loop per base.  Returns the reference's
    DataFrame (CHROM, POS, OBS, EXP, PVAL, Pi, MU, SIGMA, REGION)."""
    import pandas as pd
    from . import sequence_tools
    g = sequence_tools.get_device_genome(f_fasta)
    idx = np.asarray(idx)
    chroms = [str(c) for c in idx[:, 0]]
    starts, ends = idx[:, 1].astype(np.int64), idx[:, 2].astype(np.int64)
    if np.any((starts > 0) & (starts < n_up)):
        raise ValueError("start out of range")
    cidx = g.chrom_indices(["chr{}".format(c) for c in chroms], prefix="")
    m_chrom, m_start = _mutation_starts(f_tabix)
    name_to_idx = {str(n).replace("chr", "", 1): i for i, n in enumerate(g.names)}
    keep = np.array([c in name_to_idx for c in m_chrom], dtype=bool)
    m_cidx = np.array([name_to_idx[c] for c in m_chrom[keep]], dtype=np.int32)
    mu = np.asarray(mu_lst, dtype=np.float64)
    sigma = np.asarray(sigma_lst, dtype=np.float64)
    out = kernels.position_test(g, cidx, starts, ends, mu, sigma,
                                sequence_tools._s_prob_table(d_pr, n_up, n_down, collapse), m_cidx, m_start[keep],
                                n_up=n_up, n_down=n_down, binsize=binsize)
    nb = np.diff(out["bin_ptr"])
    rep = lambda v: np.repeat(np.asarray(v), nb)
    # an object array keeps 'X' a string and '3' an int in one column (a plain array would make every label a string)
    df = pd.DataFrame({"CHROM": rep(np.array([int(c) if c.isdigit() else c for c in chroms], dtype=object)),
                       "POS": out["pos"].cpu().numpy(), "OBS": out["obs"].cpu().numpy().astype(np.float64),
                       "EXP": out["exp"].cpu().numpy(), "PVAL": out["pval"].cpu().numpy(),
                       "Pi": out["pt"].cpu().numpy(), "MU": rep(mu), "SIGMA": rep(sigma)})
    df["REGION"] = rep(["{}:{}-{}".format(c, s, e) for c, s, e in zip(chroms, starts, ends)])
    return df


def apply_nb_to_region(CHROM, START, END, mu, sigma, S_probs, tabix, fasta, n_up=2, n_down=2, binsize=1,
                       collapse=False):
    """One region of nb_model (reference :126-186): returns (pvals, poss, obss, exps, pt_lst)."""
    df = nb_model(S_probs, np.array([[CHROM, START, END]], dtype=object), [mu], [sigma], tabix, fasta, n_up=n_up,
                  n_down=n_down, binsize=binsize, collapse=collapse)
    return (df.PVAL.values, df.POS.values, df.OBS.values.astype(np.int64), df.EXP.values, list(df.Pi.values))
