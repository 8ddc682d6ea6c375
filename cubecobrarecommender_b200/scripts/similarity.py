"""Drop-in for reference ``src/scripts/similarity.py``.

    python -m cubecobrarecommender_b200.scripts.similarity card_name N
    python -m cubecobrarecommender_b200.scripts.similarity --table N OUT.npz [--exclude-self]

``card_name`` with underscores for spaces (reference similarity.py:8).  Prints ``"{rank}: {name} {dist}"`` for the
``N`` nearest cards by the Keras ``CosineSimilarity`` loss (= -cosine) between encoder embeddings, most similar first
(the card itself leads with -1.0), like similarity.py:31-35.  The reference encodes a dense C x C identity and calls the
loss C times in a Python loop; here the embeddings come from the embedding-bag encoder and one kernel computes all C
distances.

``--table``: the similar-cards table of every card at once (``MLRecommender.similar_cards(None, N)``), written to
``OUT.npz`` as ``ids`` int32 (C, N) and ``dists`` float32 (C, N), row c the N nearest cards of card c in ``similar``'s
order; ``--exclude-self`` leaves each card out of its own row.  Prints one summary line.
"""
import sys


def parse_args(args):
    """``("card", name, n)`` for the reference form, ``("table", n, out_path, exclude_self)`` for ``--table``."""
    if args and args[0] == "--table":
        rest = [a for a in args[1:] if a != "--exclude-self"]
        if len(rest) != 2:
            raise SystemExit("usage: similarity --table N OUT.npz [--exclude-self]")
        return "table", int(rest[0]), rest[1], "--exclude-self" in args[1:]
    return "card", args[0].replace('_', ' '), int(args[1])


def main(argv=None, model_dir='ml_files/high_req', id_map='ml_files/recommender_id_map.json'):
    from ..ml.inference import MLRecommender
    from ..ml.model import load_model
    from .common import load_int_to_card
    args = sys.argv[1:] if argv is None else argv
    parsed = parse_args(args)
    if parsed[0] == "table":
        import numpy as np
        _, n, path, exclude_self = parsed
        rec = MLRecommender(load_model(model_dir))
        ids, dists = rec.similar_cards(None, n, exclude_self=exclude_self)
        ids, dists = ids.cpu().numpy(), dists.cpu().numpy()
        np.savez(path, ids=ids, dists=dists)
        print(f"similar-cards table: {ids.shape[0]} cards x {ids.shape[1]} neighbours"
              f"{' (self excluded)' if exclude_self else ''} -> {path}")
        return ids, dists
    _, name, n = parsed
    int_to_card, card_to_int = load_int_to_card(id_map)
    rec = MLRecommender(load_model(model_dir))
    ids, dists = rec.similar(card_to_int[name], n)
    out = []
    for i, (card_idx, d) in enumerate(zip(ids, dists)):
        print(str(i + 1) + ":", int_to_card[int(card_idx)], float(d))
        out.append((int_to_card[int(card_idx)], float(d)))
    return out


if __name__ == "__main__":
    main()
