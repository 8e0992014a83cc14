"""Regenerates mrqa_harness_turns.json for tests/test_e2e_tooling.py: what the unmodified multi-round-QA
harness of production-stack (benchmarks/multi-round-qa/multi-round-qa.py) sends to tools/mock_backend.py,
per (user id, number of messages): sha1 of the `messages`, max_tokens, stream.

    python tests/golden/make_harness_golden.py <production-stack checkout>/benchmarks/multi-round-qa/multi-round-qa.py
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from tests.test_e2e_tooling import HARNESS_GOLDEN, HARNESS_SHAPE, by_turn, run_against_mock  # noqa: E402


def main():
    harness = os.path.abspath(sys.argv[1])
    args = [*HARNESS_SHAPE, "--num-rounds", "3", "--time", "7", "--request-with-user-id"]
    with tempfile.TemporaryDirectory() as tmp:
        rows = run_against_mock(lambda port: [sys.executable, harness, *args, "--base-url", f"http://127.0.0.1:{port}/v1",
                                              "--output", "ref.csv"], tmp)
    turns = sorted(([u, n, *v] for (u, n), v in by_turn(rows).items()), key=lambda t: (int(t[0]), t[1]))
    with open(HARNESS_GOLDEN, "w") as f:
        f.write('{"harness_args": %s,\n "turns": [\n  %s\n ]}\n' % (json.dumps(args), ",\n  ".join(json.dumps(t) for t in turns)))
    print(f"{len(turns)} turns of {len({t[0] for t in turns})} users -> {HARNESS_GOLDEN}")


if __name__ == "__main__":
    main()
