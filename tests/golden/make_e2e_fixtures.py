#!/usr/bin/env python
"""Generates tests/golden/e2e_cases.json from the reference's own end-to-end measure cases
(<banyandb>/test/cases/measure/data/{input,want,testdata} + pkg/test/measure/testdata/measures): the data points
the integration suite writes, the query of each case and the rows it expects.  Only cases inside the hot path are
taken (group-by + aggregation, optional Top / tag filter).  The JSON it writes is the committed fixture, so the
tests need no checkout of BanyanDB.

    python tests/golden/make_e2e_fixtures.py <banyandb checkout>
"""
import json
import os
import sys

import yaml

# case -> data file written by test/cases/init.go:88,105 for that measure (group sw_metric)
CASES = {
    "float_top_mean": "service_instance_float_metric_data.json",
    "float_top_sum": "service_instance_float_metric_data.json",
    "float_top_count": "service_instance_float_metric_data.json",
    "group_count": "service_cpm_minute_data.json",
    "group_max": "service_cpm_minute_data.json",
    "group_mean": "service_cpm_minute_data.json",
    "group_min": "service_cpm_minute_data.json",
    "group_sum": "service_cpm_minute_data.json",
    "group_sum_with_filter": "service_cpm_minute_data.json",
    "top": "service_cpm_minute_data.json",
    # generated feature combinations of the same suite: order-by direction x top x filter; they also project a non-key
    # tag (entity_id), which carries the first-seen value of the group in scan order
    "gen_feat_count_group_order_desc_8": "service_cpm_minute_data.json",
    "gen_feat_max_group_order_desc_6": "service_cpm_minute_data.json",
    "gen_feat_mean_group_2": "service_cpm_minute_data.json",
    "gen_feat_mean_group_order_asc_5": "service_cpm_minute_data.json",
    "gen_feat_mean_top_asc_group_order_asc_4": "service_cpm_minute_data.json",
    "gen_feat_mean_top_asc_group_order_desc_filter_1": "service_cpm_minute_data.json",
    "gen_feat_mean_top_desc_group_order_asc_0": "service_cpm_minute_data.json",
    "gen_feat_mean_top_desc_group_order_desc_3": "service_cpm_minute_data.json",
    "gen_feat_min_group_order_desc_7": "service_cpm_minute_data.json",
    "gen_feat_sum_group_order_desc_9": "service_cpm_minute_data.json",
}


def scalar(v):
    (kind, body), = v.items()
    val = body.get("value") if isinstance(body, dict) else None
    if kind == "int":
        return {"type": "int", "value": int(val if val is not None else 0)}
    if kind == "float":
        return {"type": "float", "value": float(val if val is not None else 0.0)}
    if kind == "str":
        return {"type": "str", "value": "" if val is None else str(val)}
    raise ValueError(kind)


def main():
    ref = sys.argv[1]
    data_dir = os.path.join(ref, "test/cases/measure/data")
    schemas = os.path.join(ref, "pkg/test/measure/testdata/measures")
    out = {}
    for case, data_file in CASES.items():
        q = yaml.safe_load(open(os.path.join(data_dir, "input", case + ".yaml")))
        want = yaml.safe_load(open(os.path.join(data_dir, "want", case + ".yaml")))
        schema = json.load(open(os.path.join(schemas, q["name"] + ".json")))
        tags = [t["name"] for t in schema["tag_families"][0]["tags"]]
        fields = [(f["name"], f["field_type"]) for f in schema["fields"]]
        rows = []
        for dp in json.load(open(os.path.join(data_dir, "testdata", data_file))):
            tv = [scalar(t)["value"] for t in dp["tag_families"][0]["tags"]]
            fv = [scalar(f) for f in dp["fields"]]
            rows.append({"tags": tv, "fields": [f["value"] for f in fv]})
        gb = q["groupBy"]
        crit = None
        if "criteria" in q:
            c = q["criteria"]["condition"]
            crit = {"tag": c["name"], "op": c["op"], "value": scalar(c["value"])["value"]}
        top = None
        if "top" in q:
            top = {"n": int(q["top"]["number"]), "desc": q["top"]["fieldValueSort"] == "SORT_DESC"}
        wrows = []
        for dp in want.get("dataPoints", []):
            wtags = {t["key"]: scalar(t["value"])["value"] for t in dp["tagFamilies"][0]["tags"]}
            key = wtags[gb["tagProjection"]["tagFamilies"][0]["tags"][0]]
            val = scalar(dp["fields"][0]["value"])
            wrows.append({"group": key, "value": val["value"], "type": val["type"], "tags": wtags})
        out[case] = {
            "source": {"input": f"test/cases/measure/data/input/{case}.yaml", "want": f"test/cases/measure/data/want/{case}.yaml",
                       "data": f"test/cases/measure/data/testdata/{data_file}", "schema": f"pkg/test/measure/testdata/measures/{q['name']}.json"},
            "measure": q["name"], "family": schema["tag_families"][0]["name"], "tags": tags, "entity": schema["entity"]["tag_names"],
            "fields": [{"name": n, "type": "float" if t == "FIELD_TYPE_FLOAT" else "int"} for n, t in fields],
            "rows": rows,
            "query": {"group_by": gb["tagProjection"]["tagFamilies"][0]["tags"][0], "agg": q["agg"]["function"].replace("AGGREGATION_FUNCTION_", ""),
                      "field": q["agg"]["fieldName"], "top": top, "criteria": crit,
                      "order": (q.get("orderBy") or {}).get("sort"),
                      "projected_tags": q["tagProjection"]["tagFamilies"][0]["tags"]},
            "want": wrows,
        }
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "e2e_cases.json")
    json.dump(out, open(path, "w"), indent=1, sort_keys=True)
    print("wrote", path, {k: len(v["want"]) for k, v in out.items()})


if __name__ == "__main__":
    main()
