/* The keyed collective of include/bydb_gpu.h (bydb_scan_reduce_keyed: group-by on a stored tag across GPUs) driven from plain C, one
 * PROCESS per rank: every rank opens its context, sizes its mailbox with bydb_keyed_reduce_layout, the handles travel over a pipe,
 * the ranks connect (CUDA IPC between the processes) and run the collective with rotating roots, keyed and plain calls alternating;
 * the root compares the keyed answer with ONE context running bydb_scan_agg_keyed over all shards.  Every rank's tag holds a
 * different number of values, so the ranks' dictionaries differ.  usage: keyed_ranks <nranks> <ndevices>  (ranks share devices
 * round-robin).  CUDA must not be touched before fork(): the parent only forks, relays the handles and collects the exit codes. */
#define _POSIX_C_SOURCE 200809L
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/types.h>
#include <sys/wait.h>
#include <unistd.h>

#include "bydb_gpu.h"
#include "bydb_synth.h"

#define MAXR 8
#define SERIES_PER_RANK 6
#define POINTS 3000
#define GROUPS 4
#define ITERS 6
#define T0 1700000000000000000LL
#define STEP 60000000000LL

static int read_all(int fd, void *buf, size_t n) {
    char *p = buf;
    while (n) {
        ssize_t k = read(fd, p, n);
        if (k <= 0) return -1;
        p += k;
        n -= (size_t)k;
    }
    return 0;
}
static int write_all(int fd, const void *buf, size_t n) {
    const char *p = buf;
    while (n) {
        ssize_t k = write(fd, p, n);
        if (k <= 0) return -1;
        p += k;
        n -= (size_t)k;
    }
    return 0;
}

static bydb_part_image *shard_image(int r) {
    static bydb_synth_field flds[2] = {{"latency", BYDB_SYN_F_LATENCY, 0}, {"calls", BYDB_SYN_I_FLUCT, 0}};
    bydb_synth_spec sp;
    memset(&sp, 0, sizeof sp);
    sp.n_series = SERIES_PER_RANK; sp.n_points = POINTS; sp.sid0 = 1 + (uint64_t)r * SERIES_PER_RANK; sp.sid_step = 1;
    sp.t0 = T0 + (int64_t)r * POINTS * STEP; sp.t_step = STEP;  /* shards follow each other in time: one context scans them all */
    sp.n_fields = 2; sp.fields = flds; sp.seed = 4242;
    sp.region_values = 5 + (uint32_t)r; sp.region_run = 24;  /* "r0".."r<4+r>": rank r holds values no lower rank has */
    bydb_part_image *img = NULL;
    return bydb_synth_part(&sp, &img) == 0 ? img : NULL;
}
static int register_image(bydb_ctx *ctx, uint64_t id, bydb_part_image *img, bydb_part_h *h) {
    bydb_file files[16];
    uint32_t n = bydb_part_image_n_files(img);
    if (n > 16) return -1;
    for (uint32_t i = 0; i < n; ++i) {
        files[i].name = bydb_part_image_file_name(img, i);
        files[i].data = bydb_part_image_file_data(img, i, &files[i].len);
    }
    bydb_part_files pf = {n, files};
    return bydb_part_register(ctx, id, &pf, h);
}
static void fill_query(bydb_query *q, const bydb_part_h *parts, uint32_t n_parts, const uint64_t *sids, const int32_t *grp, uint64_t ns, const bydb_agg *aggs,
                       int top) {
    memset(q, 0, sizeof *q);
    q->parts = parts; q->n_parts = n_parts; q->series_ids = sids; q->series_group = grp; q->n_series = ns; q->n_groups = GROUPS;
    q->aggs = aggs; q->n_aggs = 4; q->tmin = T0 + 100 * STEP; q->tmax = T0 + (int64_t)(MAXR * POINTS - 500) * STEP;
    q->top_n = top; q->top_agg = 3; q->top_desc = 1;
}
static int same_key(const bydb_keyed_result *a, int i, const bydb_keyed_result *b, int j) {
    const uint32_t ka = (uint32_t)a->key_id[i], kb = (uint32_t)b->key_id[j];
    const uint32_t la = a->key_off[ka + 1] - a->key_off[ka], lb = b->key_off[kb + 1] - b->key_off[kb];
    return la == lb && memcmp(a->key_bytes + a->key_off[ka], b->key_bytes + b->key_off[kb], la) == 0;
}

static int rank_main(int rank, int nranks, int ndev, int to_parent, int from_parent) {
    bydb_cfg cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.device = rank % ndev;
    bydb_ctx *ctx = NULL;
    if (bydb_init(&cfg, &ctx) != 0) { fprintf(stderr, "rank %d: init: %s\n", rank, bydb_last_error()); return 2; }
    bydb_agg aggs[4] = {{"latency", BYDB_AGG_SUM, 0}, {"latency", BYDB_AGG_MAX, 0}, {"calls", BYDB_AGG_MIN, 0}, {"calls", BYDB_AGG_COUNT, 0}};
    uint64_t all_sids[MAXR * SERIES_PER_RANK];
    int32_t all_grp[MAXR * SERIES_PER_RANK];
    for (int i = 0; i < nranks * SERIES_PER_RANK; ++i) { all_sids[i] = 1 + (uint64_t)i; all_grp[i] = i % GROUPS; }
    bydb_group_key key = {"default", "region", 16, 0};
    bydb_query probe;
    fill_query(&probe, NULL, 0, all_sids, all_grp, (uint64_t)nranks * SERIES_PER_RANK, aggs, 0);
    uint64_t slot_bytes = 0;
    if (bydb_keyed_reduce_layout(&probe, &key, &slot_bytes) != 0) return 3;
    bydb_comm_handle mine, all[MAXR];
    if (bydb_comm_export(ctx, slot_bytes, nranks, &mine) != 0) { fprintf(stderr, "rank %d: export: %s\n", rank, bydb_last_error()); return 4; }
    if (write_all(to_parent, &mine, sizeof mine) || read_all(from_parent, all, sizeof(bydb_comm_handle) * (size_t)nranks)) return 5;
    if (bydb_comm_connect(ctx, rank, nranks, all) != 0) { fprintf(stderr, "rank %d: connect: %s\n", rank, bydb_last_error()); return 6; }
    bydb_part_image *img = shard_image(rank);
    bydb_part_h h = 0;
    if (!img || register_image(ctx, 1, img, &h) != 0) { fprintf(stderr, "rank %d: register: %s\n", rank, bydb_last_error()); return 7; }
    const uint64_t *my_sids = all_sids + rank * SERIES_PER_RANK;
    const int32_t *my_grp = all_grp + rank * SERIES_PER_RANK;
    int fails = 0;
    for (int iter = 0; iter < ITERS; ++iter) {  /* roots rotate, slot parities alternate, plain calls in between */
        const int root = iter % nranks, top = (iter & 1) ? 5 : 0;
        bydb_query q;
        fill_query(&q, &h, 1, my_sids, my_grp, SERIES_PER_RANK, aggs, top);
        if (iter % 3 == 2) {
            bydb_result plain;
            if (bydb_scan_reduce(ctx, &q, root, &plain) != 0) { fprintf(stderr, "rank %d iter %d: scan_reduce: %s\n", rank, iter, bydb_last_error()); return 8; }
            bydb_result_free(ctx, &plain);
        }
        bydb_keyed_result res;
        int rc = bydb_scan_reduce_keyed(ctx, &q, &key, root, &res);
        if (rc != 0) { fprintf(stderr, "rank %d iter %d: scan_reduce_keyed: %d %s\n", rank, iter, rc, bydb_last_error()); return 9; }
        if (rank != root) {
            if (res.base.n_rows != 0 || res.n_keys != 0 || res.base.stats.blocks_scanned == 0) ++fails;
            bydb_keyed_result_free(ctx, &res);
            continue;
        }
        /* the root checks the reduced rows against ONE context scanning all the shards */
        bydb_part_h hs[MAXR];
        bydb_part_image *imgs[MAXR];
        for (int r = 0; r < nranks; ++r) {
            imgs[r] = shard_image(r);
            if (!imgs[r] || register_image(ctx, 100 + (uint64_t)(iter * MAXR + r), imgs[r], &hs[r]) != 0) return 10;
        }
        bydb_query whole;
        fill_query(&whole, hs, (uint32_t)nranks, all_sids, all_grp, (uint64_t)nranks * SERIES_PER_RANK, aggs, top);
        bydb_keyed_result want;
        if (bydb_scan_agg_keyed(ctx, &whole, &key, &want) != 0) { fprintf(stderr, "whole scan: %s\n", bydb_last_error()); return 11; }
        if (res.base.n_rows != want.base.n_rows || res.base.n_rows == 0 || res.n_keys != want.n_keys || res.n_keys != 4 + nranks) ++fails;
        for (int i = 0; i < res.base.n_rows && i < want.base.n_rows; ++i) {
            if (res.base.group_id[i] != want.base.group_id[i] || res.base.rows[i] != want.base.rows[i] || !same_key(&res, i, &want, i)) ++fails;
            for (int a = 0; a < 4; ++a) {
                const int k = i * 4 + a;
                if (res.base.is_float[a] != want.base.is_float[a]) ++fails;
                if (res.base.is_float[a]) {
                    if (fabs(res.base.val_f64[k] - want.base.val_f64[k]) > 1e-12 * fabs(want.base.val_f64[k])) ++fails;
                } else if (res.base.val_i64[k] != want.base.val_i64[k]) {
                    ++fails;
                }
            }
        }
        bydb_keyed_result_free(ctx, &want);
        bydb_keyed_result_free(ctx, &res);
        for (int r = 0; r < nranks; ++r) {
            bydb_part_release(ctx, hs[r]);
            bydb_part_image_free(imgs[r]);
        }
    }
    bydb_part_release(ctx, h);
    bydb_part_image_free(img);
    bydb_shutdown(ctx);
    if (fails) fprintf(stderr, "rank %d: %d mismatches\n", rank, fails);
    return fails ? 12 : 0;
}

int main(int argc, char **argv) {
    const int nranks = argc > 1 ? atoi(argv[1]) : 2, ndev = argc > 2 ? atoi(argv[2]) : 1;
    if (nranks < 1 || nranks > MAXR || ndev < 1) return 64;
    int up[MAXR][2], down[MAXR][2];
    pid_t pids[MAXR];
    for (int r = 0; r < nranks; ++r) {
        if (pipe(up[r]) || pipe(down[r])) return 65;
        pids[r] = fork();
        if (pids[r] < 0) return 66;
        if (pids[r] == 0) {
            close(up[r][0]);
            close(down[r][1]);
            _exit(rank_main(r, nranks, ndev, up[r][1], down[r][0]));
        }
        close(up[r][1]);
        close(down[r][0]);
    }
    bydb_comm_handle all[MAXR];
    int bad = 0;
    for (int r = 0; r < nranks; ++r)
        if (read_all(up[r][0], &all[r], sizeof all[r])) bad = 1;
    for (int r = 0; r < nranks; ++r)
        if (bad || write_all(down[r][1], all, sizeof(bydb_comm_handle) * (size_t)nranks)) close(down[r][1]);
    int status = 0, worst = bad ? 67 : 0;
    for (int r = 0; r < nranks; ++r) {
        waitpid(pids[r], &status, 0);
        const int code = WIFEXITED(status) ? WEXITSTATUS(status) : 99;
        if (code) { fprintf(stderr, "rank %d exited with %d\n", r, code); worst = code; }
    }
    printf(worst ? "FAILED\n" : "OK %d ranks on %d device(s), %d keyed collective calls, roots rotated\n", nranks, ndev, ITERS);
    return worst;
}
