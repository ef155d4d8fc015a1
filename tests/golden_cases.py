"""Rebuilds a model (oracle or product) from a golden fixture and replays its protocol."""
import torch

ORACLE = {"DeepFM": "OracleDeepFM", "DCNModel": "OracleDCN", "DeepCrossingModel": "OracleDeepCrossing",
          "AFM": "OracleAFM", "FwFM": "OracleFwFM", "DIN": "OracleDIN", "BSTModel": "OracleBST"}


def build(fx, namespace, vocab_dir, oracle):
    name = ORACLE[fx["model"]] if oracle else fx["model"]
    cls = getattr(namespace, name)
    if fx["model"] == "AFM":
        return cls(fx["feature_columns"], **fx["ctor"])
    if fx["model"] == "FwFM":
        return cls(**fx["ctor"])
    return cls(vocab_dir, **fx["ctor"])


def call(model, fx, inputs):
    k = fx["model"]
    if k == "DeepFM":
        return model(inputs["category"])
    if k in ("DCNModel", "DeepCrossingModel", "AFM"):
        return model(inputs["dense"], inputs["category"])
    if k == "FwFM":
        return (model(inputs["x"]),)
    if k == "DIN":
        return model(inputs["dense"], inputs["category"], inputs["sequence"], inputs["target"])
    if k == "BSTModel":
        return model(inputs["dense"], inputs["category"], inputs["seq_feedid"], inputs["seq_length"])
    raise KeyError(k)


def replay(model, fx, inputs, cotangents):
    """The protocol of tests/golden/make_golden.py: seed, forward, loss = sum <out, cot>, backward."""
    model.train()
    torch.manual_seed(fx["seed"])
    outs = call(model, fx, inputs)
    tensors = [o for o in outs if torch.is_tensor(o)]
    loss = sum((o * c).sum() for o, c in zip(tensors, cotangents))
    model.zero_grad()
    loss.backward()
    grads = {k: p.grad for k, p in model.named_parameters() if p.grad is not None}
    return outs, grads


def to_double(obj):
    """The floating-point tensors of a fixture's inputs / cotangents in float64."""
    if torch.is_tensor(obj):
        return obj.double() if obj.is_floating_point() else obj
    if isinstance(obj, dict):
        return {k: to_double(v) for k, v in obj.items()}
    return [to_double(v) for v in obj]


def expand_sparse(entry):
    """A sparsely stored table of tests/golden/checkpoint_*.pt -> the full [height, dim] tensor
    (zeros in the rows the recorded batch never touches)."""
    if not isinstance(entry, dict):
        return entry
    full = torch.zeros(entry["height"], entry["dim"], dtype=entry["values"].dtype)
    full[entry["rows"]] = entry["values"]
    return full


def expand_checkpoint(fx):
    """In place: state_dict and grads of a checkpoint fixture as dense tensors."""
    fx["state_dict"] = {k: expand_sparse(v) for k, v in fx["state_dict"].items()}
    fx["grads"] = {k: expand_sparse(v) for k, v in fx["grads"].items()}
    return fx
