"""Host-side unit test of the tcgen05 GEMM's persistent tile schedule (csrc/tc_sched.h — the same functions the kernel
calls, compiled here with g++): for every shape, every output element of the [num_m*128, N] result is produced by
exactly one unit of work, every CTA's work list is the same for its three warp roles by construction, half tiles appear
only in the last round and only where the host enabled them, and the last-wave split never makes the longest CTA longer.
The launch plan (tc_nt_plan, with the default knobs) keeps the invariants the kernel relies on over a grid of shapes."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = os.path.join(ROOT, "normalizing-flow-with-diffusion-prior-model_b200", "csrc")

HARNESS = r"""
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "tc_sched.h"
using namespace nfdpm;
int main(int argc, char** argv) {
  const int grids[] = {1, 2, 7, 64, 132, 148};
  const int bns[] = {16, 64, 112, 128, 256};
  long long cases = 0, split_cases = 0;
  for (int grid_sms : grids)
    for (int BN : bns)
      for (int num_n = 1; num_n <= 4; ++num_n)
        for (int num_m = 1; num_m <= 300; num_m += (num_m < 40 ? 1 : 37)) {
          const int N = num_n * BN, tiles = num_m * num_n, grid = tiles < grid_sms ? tiles : grid_sms;
          for (int want_split = 0; want_split <= 1; ++want_split) {
            const int split = want_split && tc_split_ok(tiles, grid, BN, N);
            if (want_split && !split) continue;
            ++cases; split_cases += split;
            std::vector<int> cover((size_t)num_m * N, 0);
            long long longest = 0;                       // in half-tile units
            for (int cta = 0; cta < grid; ++cta) {
              TcWork w; long long cost = 0; int it = 0, seen_half = 0;
              for (; tc_work_for(cta, grid, it, tiles, num_n, BN, split, w); ++it) {
                if (w.bn != BN) {
                  if (!split || w.bn * 2 != BN || (w.bn % 64) != 0) { printf("bad half tile\n"); return 1; }
                  seen_half = 1; cost += 1;
                } else {
                  if (seen_half) { printf("full tile after a half tile\n"); return 1; }
                  cost += 2;
                }
                if (w.m_blk < 0 || w.m_blk >= num_m || w.n0 < 0 || w.n0 + w.bn > N) { printf("out of range\n"); return 1; }
                for (int c = 0; c < w.bn; ++c) cover[(size_t)w.m_blk * N + w.n0 + c] += 1;
              }
              TcWork w2;                                  // once exhausted, the schedule stays exhausted
              if (tc_work_for(cta, grid, it + 1, tiles, num_n, BN, split, w2)) { printf("not exhausted\n"); return 1; }
              if (cost > longest) longest = cost;
            }
            for (int v : cover) if (v != 1) { printf("coverage %d (grid %d BN %d num_n %d num_m %d split %d)\n", v, grid, BN, num_n, num_m, split); return 1; }
            const long long unsplit_longest = 2LL * ((tiles + grid - 1) / grid);
            if (longest > unsplit_longest) { printf("split made the longest CTA longer\n"); return 1; }
            if (split && longest >= unsplit_longest) { printf("split did not shorten the last wave\n"); return 1; }
          }
        }
  // the case the split was written for: M = 32768, N = 512, BN = 256 on 148 SMs
  if (!tc_split_ok(512, 148, 256, 512)) { printf("headline shape not split\n"); return 1; }
  printf("ok %lld cases, %lld split\n", cases, split_cases);
  return 0;
}
"""


def test_tile_schedule_covers_every_output_exactly_once(tmp_path):
    src = tmp_path / "sched.cpp"
    src.write_text(HARNESS)
    exe = tmp_path / "sched"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-I", HDR, str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:]
    assert r.stdout.startswith("ok") and int(r.stdout.split()[3]) > 0, r.stdout


PLAN_HARNESS = r"""
#include <cstdio>
#include "tc_sched.h"
using namespace nfdpm;
#define FAIL(msg) do { printf("%s: M %d N %d Kmem %d out %d actnorm %d sms %d BN %d split %d stages %d smem %d\n", msg, M, N, \
                              Kmem, out, (int)act, sms, p.BN, p.split, p.plan.n_stages, p.smem); return 1; } while (0)
int main() {
  const int Ms[] = {1, 77, 128, 129, 300, 2048, 4096, 8192, 32768, 50000, 131072};
  const int Ks[] = {64, 128, 192, 256, 512, 1024, 2048};
  const int smss[] = {148, 132, 8};
  long long cases = 0, deep = 0, split = 0, narrowed = 0;
  for (int sms : smss)
    for (int M : Ms)
      for (int N = 16; N <= 4096; N += (N < 1024 ? 16 : 112))
        for (int Kmem : Ks)
          for (int out = 0; out < 3; ++out)                     // 0 fp32, 1 bf16, 2 split pairs
            for (int a = 0; a < 2; ++a) {
              const bool act = a == 1, f32 = out == 0, bf16 = out == 1;
              if (out == 2 && N % 32) continue;                 // split-pair rows hold whole groups of 32 columns
              if (act && N > 2048) continue;                    // the fused ActNorm epilogue supports N <= 2048
              const TcNtPlan p = tc_nt_plan(M, N, Kmem, f32, bf16, act, sms, 256, 74, 1, 1);
              ++cases;
              const int cpb = bf16 ? 64 : 32;
              if (p.BN > 256 || p.BN % 16 || p.BN < 16) FAIL("BN out of range");
              if (f32 && p.BN > 128) FAIL("fp32 output BN > 128");
              if (p.num_n > 1 && p.BN % cpb) FAIL("several N blocks, BN not whole store boxes");
              if (p.num_n * p.BN < N || (p.num_n - 1) * p.BN >= N) FAIL("N blocks do not cover N exactly");
              if (p.tiles != (M + TC_BM - 1) / TC_BM * p.num_n) FAIL("tile count");
              if (p.grid != (p.tiles < sms ? p.tiles : sms)) FAIL("grid");
              if (p.plan.n_stages < 2 || p.plan.n_stages > TC_MAX_STAGES) FAIL("n_stages out of range");
              if (p.smem > TC_SMEM_MAX) FAIL("shared memory over 226 KB");
              if (p.split && !tc_split_ok(p.tiles, p.grid, p.BN, N)) FAIL("split without tc_split_ok");
              const int extra = act ? 2 * p.num_n * p.BN * 4 : 0;
              if (p.smem != 1024 + p.plan.n_stages * p.plan.stage_bytes + p.plan.cstage_bytes + extra) FAIL("smem sum");
              if (p.plan.stage_bytes < TC_A_BYTES + p.BN * TC_BK * 2) FAIL("stage smaller than its boxes");
              // the staging buffer holds what one pass of the epilogue stores
              const int pass_cols = p.plan.cpw * 64 < p.BN ? p.plan.cpw * 64 : p.BN;
              if (p.plan.cstage_bytes < 128 * pass_cols * (bf16 ? 2 : 4)) FAIL("staging smaller than one pass");
              if (p.plan.cpw == 1 ? p.plan.cstage_bytes != 128 * 64 * (bf16 ? 2 : 4) : p.plan.cstage_bytes != TC_CSTAGE_BYTES)
                FAIL("staging size");
              deep += p.plan.cpw == 1; split += p.split;
              narrowed += p.BN < (N < (f32 ? 128 : 256) ? N : (f32 ? 128 : 256)) && p.num_n > 1;
            }
  printf("ok %lld cases, %lld deep, %lld split, %lld narrowed\n", cases, deep, split, narrowed);
  return (deep && split && narrowed) ? 0 : 1;
}
"""


def test_launch_plan_invariants(tmp_path):
    src = tmp_path / "plan.cpp"
    src.write_text(PLAN_HARNESS)
    exe = tmp_path / "plan"
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-I", HDR, str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("ok"), r.stdout[-2000:]
