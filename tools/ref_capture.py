"""Run the real reference generator while recording every torch.rand/randn draw
(TEST INFRASTRUCTURE: the golden generators record the reference's draws with it; the tests
replay them through draws_from_log)."""
import contextlib
import torch


@contextlib.contextmanager
def record_draws(log):
    orig_rand, orig_randn = torch.rand, torch.randn

    def rand(*a, **k):
        t = orig_rand(*a, **k)
        log.append(("rand", t.clone()))
        return t

    def randn(*a, **k):
        t = orig_randn(*a, **k)
        log.append(("randn", t.clone()))
        return t

    torch.rand, torch.randn = rand, randn
    try:
        yield log
    finally:
        torch.rand, torch.randn = orig_rand, orig_randn


def draws_from_log(log, hierarchical=True):
    """Map the whole_grad_forward (forward_points=None) draw order to named tensors
    (SURVEY.md §7 hard part 4)."""
    it = iter(log)
    d = {}
    k, t = next(it); assert k == "rand"; d["jitter_u"] = t[..., 0]
    k, t = next(it); assert k == "randn"; d["yaw_n"] = t
    k, t = next(it); assert k == "randn"; d["pitch_n"] = t
    if hierarchical:
        k, t = next(it); assert k == "randn"; d["noise_c"] = t[..., 0]
        k, t = next(it); assert k == "rand"; d["pdf_u"] = t
    k, t = next(it); assert k == "randn"; d["noise_f"] = t[..., 0]
    return d
