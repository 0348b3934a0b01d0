"""Records tests/golden/elements_branches_golden.npz by RUNNING THE REFERENCE ITSELF (read-only upstream tree, found like
make_golden.py finds it: SAT_REFERENCE_DIR, else /root/reference).

    python tests/golden/make_golden_branches.py

calculate_orbital_elements on its circular (satellite_function.py:212, :223-227) and parabolic (:186-190, :247-253)
branches, and calculate_state_information on its 5- and 4-element forms (:287-315). Candidate states are drawn by
tests/elements_forms.py and the reference itself decides which branch each takes; nothing stored here comes from the
oracle or from the CUDA path.
"""
from __future__ import annotations

import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import elements_forms as F  # noqa: E402
import refshim  # noqa: E402

warnings.filterwarnings("ignore")
MU = 3.986e14


def main():
    T = refshim.load()["satellite_function"].Time_window_of_danger_zone

    class Ref:                                              # the interface elements_forms' searches call
        @staticmethod
        def orbital_elements(miu, R, V):
            return T.calculate_orbital_elements(miu, np.asarray(R, dtype=np.float64), np.asarray(V, dtype=np.float64))

    rng = np.random.default_rng(2024)
    circ = F.circular_states(rng, Ref, 96)
    circ_eq = F.circular_states(rng, Ref, 32, equatorial=True)
    para = F.parabolic_states(rng, Ref, 96)
    near = F.near_miss_states(Ref, np.concatenate([circ, circ_eq]), para)
    rv = np.concatenate([circ, circ_eq, para, near])
    tag = np.concatenate([np.full(len(circ), 0), np.full(len(circ_eq), 1), np.full(len(para), 2), np.full(len(near), 3)])
    elements = np.zeros((len(rv), 6))
    kind = np.zeros(len(rv), dtype=np.int32)
    for k in range(len(rv)):
        el = Ref.orbital_elements(MU, rv[k, :3], rv[k, 3:])
        elements[k, :len(el)] = el
        kind[k] = len(el)
    # every 5- and 4-element input form: random sets with special angles, and the lists the branches above returned
    form5 = np.concatenate([F.five_forms(rng, 256), elements[kind == 5, :5]])
    form4 = np.concatenate([F.four_forms(rng, 256), elements[kind == 4, :4]])
    state5 = np.array([np.concatenate(T.calculate_state_information(list(r), miu=MU)) for r in form5])
    state4 = np.array([np.concatenate(T.calculate_state_information(list(r), miu=MU)) for r in form4])
    path = os.path.join(HERE, "elements_branches_golden.npz")
    np.savez_compressed(path, rv=rv, tag=tag, elements=elements, kind=kind, form5=form5, state5=state5,
                        form4=form4, state4=state4)
    print(f"wrote {path} [{os.path.getsize(path) / 1024:.0f} KiB]")


if __name__ == "__main__":
    if not refshim.available():
        sys.exit(f"the upstream reference tree is not at {refshim.REF} (set SAT_REFERENCE_DIR)")
    main()
